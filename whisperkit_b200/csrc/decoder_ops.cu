// Decoder-side kernels: everything one autoregressive step needs besides the (swap-AB, split-K) tcgen05 GEMMs.
//
// Reference behaviour restated on the device (so the host sees only final token IDs):
//   decodeText loop state machine            Sources/WhisperKit/Core/TextDecoder.swift:566-686
//   updateKVCache (host splice, eliminated)  Sources/WhisperKit/Core/TextDecoder.swift:218-270
//   LogitsFiltering x4                       Sources/WhisperKit/Core/Text/LogitsFilter.swift:12-276
//   GreedyTokenSampler.update                Sources/WhisperKit/Core/Text/TokenSampler.swift:42-83,215-240
#include <curand_kernel.h>
#include <math.h>

#include <stdlib.h>

#include "common.cuh"
#include <algorithm>
#include "kernels.h"

namespace wk {

static constexpr int kMaxCtx = 224;  // Constants.maxTokenContext (Models.swift:1334)

__device__ __forceinline__ float block_sum(float v, float* scratch) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    float r = (lane < nw) ? scratch[lane] : 0.f;
    r = warp_sum(r);
    return r;
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
    v = warp_max(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    float r = (lane < nw) ? scratch[lane] : -INFINITY;
    r = warp_max(r);
    return r;
}

// =====================================================================================================
// decode state
// =====================================================================================================
__global__ void decode_slots_init_kernel(DecodeState st, RowParams* __restrict__ rp_dev, const int32_t* __restrict__ slot_ids,
                                         const int32_t* __restrict__ prompts, const RowParams* __restrict__ rp_new, BeamState bs) {
    const int i = blockIdx.x, b = slot_ids[i];
    const RowParams R = rp_new[i];
    const int n_prompt = R.prompt_len;
    for (int t = threadIdx.x; t < kMaxCtx; t += blockDim.x) {
        st.tokens[b * kMaxCtx + t] = t < n_prompt ? prompts[i * kMaxCtx + t] : 0;
        st.logprobs[b * kMaxCtx + t] = 0.f;
    }
    if (threadIdx.x == 0) {
        rp_dev[b] = R;
        st.n_tokens[b] = n_prompt;
        st.next_token[b] = n_prompt > 0 ? prompts[i * kMaxCtx + n_prompt - 1] : 0;
        st.done[b] = 0;
        st.first_low[b] = 0;
        st.steps[b] = 0;
        st.input_ids[b] = 0;
        st.error[b] = 0;
        st.lang_tok[b] = -1;
        st.lang_lp[b] = 0.f;
        if (bs.beam > 1) {
            bs.sum_lp[b] = 0.f;
            if (b % bs.beam == 0) bs.n_fin[b / bs.beam] = 0;
        }
    }
}

wk_status decode_slots_init(DecodeState st, RowParams* rp_dev, const int32_t* slot_ids, const int32_t* prompts, const RowParams* rp_new,
                            int n, cudaStream_t stream, BeamState beam) {
    if (n < 1) return WK_OK;
    decode_slots_init_kernel<<<n, 64, 0, stream>>>(st, rp_dev, slot_ids, prompts, rp_new, beam);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decode_slots_init launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

// =====================================================================================================
// token + position embedding, prompt forcing (TextDecoder.swift:581-594), first LayerNorm
// =====================================================================================================
template <typename T>
__global__ void __launch_bounds__(256)
decoder_embed_ln_kernel(const T* __restrict__ emb, const float* __restrict__ pos_emb, const float* __restrict__ gamma,
                        const float* __restrict__ beta, DecodeState st, int vocab, int ts_begin, int sot, float* __restrict__ x,
                        T* __restrict__ xn, int d, const int32_t* __restrict__ explicit_pos) {
    __shared__ float scratch[32];
    const int b = blockIdx.x, tid = threadIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    int tok, pos;
    if (explicit_pos) {
        tok = st.input_ids[b];
        pos = explicit_pos[b];
    } else {
        if (st.done[b]) return;          // the window has ended: its row of the step is dead (x / xn keep their last values)
        const int step = st.steps[b];
        const int prompt_len = st.rp[b].prompt_len;
        pos = step;
        tok = st.next_token[b];
        bool overwrite = false;
        if (step == 0 && (st.rp[b].lang_flags & kLangPreStep) && st.lang_tok[b] < 0) {
            tok = sot;                   // language-detection pre-step: SOT at position 0 (the prompt's own step 0 overwrites its K/V row)
        } else if (step < prompt_len) {
            const int cur = st.tokens[b * kMaxCtx + step];
            const bool is_ts = cur >= ts_begin, pred_ts = tok >= ts_begin;
            if (!(step == prompt_len - 1 && is_ts && pred_ts)) tok = cur;
            else overwrite = true;  // model-predicted first timestamp replaces the forced <|0.00|>
        }
        __syncthreads();
        if (tid == 0) {
            if (overwrite) st.tokens[b * kMaxCtx + step] = tok;
            st.input_ids[b] = tok;
        }
    }
    tok = min(max(tok, 0), vocab - 1);   // never index the embedding table out of bounds
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = tid + k * 256;
        v[k] = 0.f;
        if (i < d) {
            v[k] = T16<T>::to_f(emb[(long long)tok * d + i]) + pos_emb[(long long)pos * d + i];
            x[(long long)b * d + i] = v[k];
            s += v[k];
        }
    }
    const float mean = block_sum(s, scratch) / d;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = tid + k * 256;
        if (i < d) { const float a = v[k] - mean; q += a * a; }
    }
    const float rstd = rsqrtf(block_sum(q, scratch) / d + 1e-5f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int i = tid + k * 256;
        if (i < d) xn[(long long)b * d + i] = T16<T>::from_f((v[k] - mean) * rstd * gamma[i] + beta[i]);
    }
}

wk_status decoder_embed_ln(const void* emb16, const float* pos, const float* gamma, const float* beta, DecodeState st, int vocab,
                           int ts_begin, int sot, float* x, void* xn, int B, int d, int dtype, const int32_t* explicit_pos, cudaStream_t stream) {
    if (d > 2048) { set_error("decoder_embed_ln: d_model %d > 2048", d); return WK_ERR_INVALID_ARGUMENT; }
    if (dtype == WK_DTYPE_F16)
        launch_k(decoder_embed_ln_kernel<__half>, dim3(B), dim3(256), 0, stream, 1, (const __half*)emb16, pos, gamma, beta, st, vocab, ts_begin, sot, x, (__half*)xn, d, explicit_pos);
    else
        launch_k(decoder_embed_ln_kernel<__nv_bfloat16>, dim3(B), dim3(256), 0, stream, 1, (const __nv_bfloat16*)emb16, pos, gamma, beta, st, vocab, ts_begin, sot, x, (__nv_bfloat16*)xn, d, explicit_pos);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_embed_ln launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

// =====================================================================================================
// split-K reduce + bias + residual + LayerNorm      (partials [S][Bp][d] f32, written by the swap-AB GEMM)
// =====================================================================================================
static constexpr int kReduceThreads = 320;   // one float4 per thread at d = 1280
static constexpr int kMaxSplits = 20;

// All split-K partial loads of a thread are issued back to back (fully unrolled, predicated) so the kernel pays one
// L2 round trip instead of `splits` serial ones; the sum runs in a fixed order (deterministic).
template <typename T>
__global__ void __launch_bounds__(kReduceThreads)
decoder_reduce_resid_ln_kernel(const float* __restrict__ partial, int splits, int Bp, const float* __restrict__ bias,
                               const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ x,
                               T* __restrict__ xn, int d) {
    __shared__ float scratch[32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int d4 = d >> 2;
    pdl_launch_dependents();
    pdl_wait();
    float4 v[2];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i4 = tid + k * kReduceThreads;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i4 < d4) {
            float4 p[kMaxSplits];
#pragma unroll
            for (int sp = 0; sp < kMaxSplits; ++sp)
                if (sp < splits) p[sp] = __ldcg(reinterpret_cast<const float4*>(partial + ((long long)sp * Bp + b) * d) + i4);
            float4 a = reinterpret_cast<const float4*>(x + (long long)b * d)[i4];
            if (bias) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(bias) + i4);
                a.x += bb.x; a.y += bb.y; a.z += bb.z; a.w += bb.w;
            }
#pragma unroll
            for (int sp = 0; sp < kMaxSplits; ++sp)
                if (sp < splits) { a.x += p[sp].x; a.y += p[sp].y; a.z += p[sp].z; a.w += p[sp].w; }
            v[k] = a;
            reinterpret_cast<float4*>(x + (long long)b * d)[i4] = a;
            s += a.x + a.y + a.z + a.w;
        }
    }
    const float mean = block_sum(s, scratch) / d;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i4 = tid + k * kReduceThreads;
        if (i4 < d4) {
            const float a0 = v[k].x - mean, a1 = v[k].y - mean, a2 = v[k].z - mean, a3 = v[k].w - mean;
            q += a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3;
        }
    }
    const float rstd = rsqrtf(block_sum(q, scratch) / d + 1e-5f);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i4 = tid + k * kReduceThreads;
        if (i4 < d4) {
            const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i4), bb = __ldg(reinterpret_cast<const float4*>(beta) + i4);
            uint2 pk;
            pk.x = T16<T>::pack2((v[k].x - mean) * rstd * g.x + bb.x, (v[k].y - mean) * rstd * g.y + bb.y);
            pk.y = T16<T>::pack2((v[k].z - mean) * rstd * g.z + bb.z, (v[k].w - mean) * rstd * g.w + bb.w);
            reinterpret_cast<uint2*>(xn + (long long)b * d)[i4] = pk;
        }
    }
}

wk_status decoder_reduce_resid_ln(const float* partial, int splits, int Bp, const float* bias, const float* gamma,
                                  const float* beta, float* x, void* xn, int B, int d, int dtype, cudaStream_t stream) {
    if (splits > kMaxSplits || d > 8 * kReduceThreads || (d & 3)) {
        set_error("decoder_reduce_resid_ln: unsupported splits %d / d %d", splits, d);
        return WK_ERR_INVALID_ARGUMENT;
    }
    if (dtype == WK_DTYPE_F16)
        launch_k(decoder_reduce_resid_ln_kernel<__half>, dim3(B), dim3(kReduceThreads), 0, stream, 32, partial, splits, Bp, bias, gamma, beta, x, (__half*)xn, d);
    else
        launch_k(decoder_reduce_resid_ln_kernel<__nv_bfloat16>, dim3(B), dim3(kReduceThreads), 0, stream, 32, partial, splits, Bp, bias, gamma, beta, x, (__nv_bfloat16*)xn, d);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_reduce_resid_ln launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

template <typename T>
__global__ void __launch_bounds__(256)
decoder_reduce_bias_gelu_kernel(const float* __restrict__ partial, int splits, int Bp, const float* __restrict__ bias,
                                T* __restrict__ out, int B, int n) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (idx >= (long long)B * n) return;
    const int b = (int)(idx / n), i = (int)(idx - (long long)b * n);
    float4 a = *reinterpret_cast<const float4*>(bias + i);
    float4 p[8];
#pragma unroll
    for (int sp = 0; sp < 8; ++sp)
        if (sp < splits) p[sp] = __ldcg(reinterpret_cast<const float4*>(partial + ((long long)sp * Bp + b) * n + i));
#pragma unroll
    for (int sp = 0; sp < 8; ++sp)
        if (sp < splits) { a.x += p[sp].x; a.y += p[sp].y; a.z += p[sp].z; a.w += p[sp].w; }
    for (int sp = 8; sp < splits; ++sp) {
        const float4 pp = __ldcg(reinterpret_cast<const float4*>(partial + ((long long)sp * Bp + b) * n + i));
        a.x += pp.x; a.y += pp.y; a.z += pp.z; a.w += pp.w;
    }
    uint2 pk;
    pk.x = T16<T>::pack2(gelu_erf(a.x), gelu_erf(a.y));
    pk.y = T16<T>::pack2(gelu_erf(a.z), gelu_erf(a.w));
    *reinterpret_cast<uint2*>(out + (long long)b * n + i) = pk;
}

wk_status decoder_reduce_bias_gelu(const float* partial, int splits, int Bp, const float* bias, void* out, int B, int n,
                                   int dtype, cudaStream_t stream) {
    const long long threads = (long long)B * n / 4;
    const unsigned grid = (unsigned)((threads + 255) / 256);
    if (dtype == WK_DTYPE_F16)
        launch_k(decoder_reduce_bias_gelu_kernel<__half>, dim3(grid), dim3(256), 0, stream, 32, partial, splits, Bp, bias, (__half*)out, B, n);
    else
        launch_k(decoder_reduce_bias_gelu_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, 32, partial, splits, Bp, bias, (__nv_bfloat16*)out, B, n);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_reduce_bias_gelu launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

// =====================================================================================================
// self attention for one new token: one CTA (4 warps) per (b, h).  Warp 0 reduces the q/k/v split-K partials and appends K/V in place
// in the device cache (replaces the host-side updateKVCache splice); the cached positions are then split over the 4 warps - 8 lanes
// per 128-byte row, 4 rows per warp instruction, several instructions in flight - so that B*H*4 warps keep enough loads in the air
// for what is a latency-bound gather (<= 223 rows of K and of V per head).  cache layout [B][H][max_len][64]
// =====================================================================================================
template <typename T, bool kAnc>
__global__ void __launch_bounds__(128)
decoder_self_attention_kernel(const float* __restrict__ partial, int splits, int Bp, const float* __restrict__ bq,
                              const float* __restrict__ bv, T* __restrict__ kcache, T* __restrict__ vcache,
                              const int32_t* __restrict__ pos_ptr, const int32_t* __restrict__ done,
                              T* __restrict__ out, int B, int H, int max_len, const int32_t* __restrict__ anc) {
    __shared__ float sq[64], skc[64], svc[64];
    __shared__ float sp[kMaxCtx];
    __shared__ float red[4][64];
    __shared__ float sstat[8];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int bh = blockIdx.x, b = bh / H, h = bh % H;
    pdl_launch_dependents();
    pdl_wait();
    if (done != nullptr && done[b]) return;   // ended window: no cache traffic
    const int dm = H * 64;
    const int pos = pos_ptr[b];
    // cache row of position t: this sequence's own row, or (beam search) the row of the ancestor beam that produced position t
    const int32_t* arow = kAnc ? anc + (long long)b * max_len : nullptr;
    const long long own = (long long)bh * max_len;
    auto row_of = [&](int t) -> long long { return kAnc ? ((long long)arow[t] * H + h) * max_len + t : own + t; };
    if (warp == 0) {
        const int e = 2 * lane;
        float2 q = make_float2(bq[h * 64 + e], bq[h * 64 + e + 1]);
        float2 k = make_float2(0.f, 0.f);
        float2 v = make_float2(bv[h * 64 + e], bv[h * 64 + e + 1]);
        for (int s = 0; s < splits; ++s) {
            const float* pr = partial + ((long long)s * Bp + b) * (3LL * dm) + h * 64 + e;
            const float2 pq = *reinterpret_cast<const float2*>(pr);
            const float2 pk = *reinterpret_cast<const float2*>(pr + dm);
            const float2 pv = *reinterpret_cast<const float2*>(pr + 2 * dm);
            q.x += pq.x; q.y += pq.y; k.x += pk.x; k.y += pk.y; v.x += pv.x; v.y += pv.y;
        }
        // append to the cache (16-bit rounding is part of the precision policy); the new row always goes to the sequence's own cache row
        const uint32_t k16 = T16<T>::pack2(k.x, k.y), v16 = T16<T>::pack2(v.x, v.y);
        *reinterpret_cast<uint32_t*>(kcache + (own + pos) * 64 + e) = k16;
        *reinterpret_cast<uint32_t*>(vcache + (own + pos) * 64 + e) = v16;
        const float2 kr = T16<T>::unpack2(k16), vr = T16<T>::unpack2(v16);
        sq[e] = q.x; sq[e + 1] = q.y;
        skc[e] = kr.x; skc[e + 1] = kr.y;
        svc[e] = vr.x; svc[e + 1] = vr.y;
        const float self = warp_sum(q.x * kr.x + q.y * kr.y);   // the current position's score comes from registers
        if (lane == 0) sp[pos] = self * 0.125f;
    }
    __syncthreads();
    const int sub = lane & 7, rsel = lane >> 3;   // 16-byte piece of the 128-byte row / row within a group of 4
    float qv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) qv[j] = sq[sub * 8 + j];
    // ---- scores over the cached positions: warp w takes rows 16 i + 4 w + rsel
    const T* kb = kcache + sub * 8;
#pragma unroll 4
    for (int t0 = warp * 4; t0 < pos; t0 += 16) {
        const int t = t0 + rsel;
        float acc = 0.f;
        if (t < pos) {
            const uint4 u = *reinterpret_cast<const uint4*>(kb + row_of(t) * 64);
            const float2 a0 = T16<T>::unpack2(u.x), a1 = T16<T>::unpack2(u.y), a2 = T16<T>::unpack2(u.z), a3 = T16<T>::unpack2(u.w);
            acc = qv[0] * a0.x + qv[1] * a0.y + qv[2] * a1.x + qv[3] * a1.y + qv[4] * a2.x + qv[5] * a2.y + qv[6] * a3.x + qv[7] * a3.y;
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
        if (sub == 0 && t < pos) sp[t] = acc * 0.125f;
    }
    __syncthreads();
    // ---- softmax over positions 0..pos
    float mx = -INFINITY;
    for (int t = tid; t <= pos; t += 128) mx = fmaxf(mx, sp[t]);
    mx = warp_max(mx);
    if (lane == 0) sstat[warp] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(sstat[0], sstat[1]), fmaxf(sstat[2], sstat[3]));
    float sm = 0.f;
    for (int t = tid; t <= pos; t += 128) {
        const float pr = __expf(sp[t] - mx);
        sp[t] = pr;
        sm += pr;
    }
    sm = warp_sum(sm);
    if (lane == 0) sstat[4 + warp] = sm;
    __syncthreads();
    const float inv = 1.f / (sstat[4] + sstat[5] + sstat[6] + sstat[7]);
    // ---- output: sum_t p[t] V[t]
    float o8[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o8[j] = 0.f;
    const T* vb = vcache + sub * 8;
#pragma unroll 4
    for (int t0 = warp * 4; t0 < pos; t0 += 16) {
        const int t = t0 + rsel;
        if (t < pos) {
            const float pr = sp[t];
            const uint4 u = *reinterpret_cast<const uint4*>(vb + row_of(t) * 64);
            const float2 a0 = T16<T>::unpack2(u.x), a1 = T16<T>::unpack2(u.y), a2 = T16<T>::unpack2(u.z), a3 = T16<T>::unpack2(u.w);
            o8[0] += pr * a0.x; o8[1] += pr * a0.y; o8[2] += pr * a1.x; o8[3] += pr * a1.y;
            o8[4] += pr * a2.x; o8[5] += pr * a2.y; o8[6] += pr * a3.x; o8[7] += pr * a3.y;
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        o8[j] += __shfl_xor_sync(0xffffffffu, o8[j], 8);
        o8[j] += __shfl_xor_sync(0xffffffffu, o8[j], 16);
    }
    if (rsel == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[warp][sub * 8 + j] = o8[j];
    }
    __syncthreads();
    if (tid < 64) {
        // the current position comes from shared memory (its cache row was written by this CTA just above)
        const float o = red[0][tid] + red[1][tid] + red[2][tid] + red[3][tid] + sp[pos] * svc[tid];
        out[(long long)b * dm + h * 64 + tid] = T16<T>::from_f(o * inv);
    }
}

wk_status decoder_self_attention(const float* partial, int splits, int Bp, const float* bq, const float* bv, void* kcache,
                                 void* vcache, const int32_t* pos, const int32_t* done, void* out, int B, int H,
                                 int max_len, int dtype, cudaStream_t stream, const int32_t* anc) {
    if (max_len > kMaxCtx) { set_error("decoder_self_attention: max_len %d > %d", max_len, kMaxCtx); return WK_ERR_INVALID_ARGUMENT; }
    const unsigned grid = (unsigned)(B * H);
    if (dtype == WK_DTYPE_F16) {
        if (anc) launch_k(decoder_self_attention_kernel<__half, true>, dim3(grid), dim3(128), 0, stream, 2, partial, splits, Bp, bq, bv, (__half*)kcache, (__half*)vcache, pos, done, (__half*)out, B, H, max_len, anc);
        else launch_k(decoder_self_attention_kernel<__half, false>, dim3(grid), dim3(128), 0, stream, 2, partial, splits, Bp, bq, bv, (__half*)kcache, (__half*)vcache, pos, done, (__half*)out, B, H, max_len, anc);
    } else {
        if (anc) launch_k(decoder_self_attention_kernel<__nv_bfloat16, true>, dim3(grid), dim3(128), 0, stream, 2, partial, splits, Bp, bq, bv, (__nv_bfloat16*)kcache, (__nv_bfloat16*)vcache, pos, done, (__nv_bfloat16*)out, B, H, max_len, anc);
        else launch_k(decoder_self_attention_kernel<__nv_bfloat16, false>, dim3(grid), dim3(128), 0, stream, 2, partial, splits, Bp, bq, bv, (__nv_bfloat16*)kcache, (__nv_bfloat16*)vcache, pos, done, (__nv_bfloat16*)out, B, H, max_len, anc);
    }
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_self_attention launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

// =====================================================================================================
// cross attention for one query per (b, h) over T encoder positions.  HBM-streaming kernel: each CTA pulls its
// contiguous K block then V block (T x 64 x 2 B each) through a 4-deep ring of 16 KB bulk-copy stages
// (cp.async.bulk + mbarrier), a dedicated producer warp keeps the ring full while 4 consumer warps compute.
// K/V layout [B][H][T][64] (written head-major by the cross-KV GEMM epilogue).
// =====================================================================================================
static constexpr int kCrossRows = 125;              // rows per stage: 125 * 128 B = 16000 B (multiple of 16)
static constexpr int kCrossStageBytes = kCrossRows * 128;
static constexpr int kCrossStages = 4;
static constexpr int kCrossThreads = 160;           // 4 consumer warps + 1 producer warp

template <typename T>
__global__ void __launch_bounds__(kCrossThreads)
decoder_cross_attention_kernel(const float* __restrict__ partial, int splits, int Bp, const float* __restrict__ bq,
                               const T* __restrict__ kcross, const T* __restrict__ vcross, T* __restrict__ out, int B, int H,
                               int Tlen, const int32_t* __restrict__ done, float* __restrict__ align_scratch, uint32_t align_mask, int kv_div) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* ring = smem;                                                   // kCrossStages * 16000
    float* scores = reinterpret_cast<float*>(smem + kCrossStages * kCrossStageBytes);  // [Tlen]
    float* sq = scores + ((Tlen + 3) & ~3);                                 // [64]
    float* red = sq + 64;                                                   // [4][64] + scratch
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(red + 4 * 64 + 32);
    uint64_t* empty_bar = full_bar + kCrossStages;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // grid order: (window, head, beam) - the kv_div rows that share one K/V block are adjacent, so their streams meet in L2
    const int beam_j = blockIdx.x % kv_div, wh = blockIdx.x / kv_div;
    const int win = wh / H, h = wh % H, b = win * kv_div + beam_j;
    const int kvh = win * H + h;             // K/V block index: [window][head]
    const int dm = H * 64;
    const int chunks = Tlen / kCrossRows;  // per K and per V
    pdl_launch_dependents();
    // ended window: skip its 2 x 192 KB K/V stream.  done[] was written by the sampler of the previous step, many kernels upstream, so it
    // may be read before griddepcontrol.wait; the load is issued here and consumed after the barrier set-up so that its latency hides
    // under it (the CTA lives ~8 us: a dependent L2 round trip at its start would cost several per cent of the kernel)
    const int ended = done != nullptr ? done[b] : 0;
    if (tid == 0) {
        for (int i = 0; i < kCrossStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 4); }
        fence_barrier_init();
    }
    __syncthreads();
    if (ended) { pdl_wait(); return; }   // (the wait still runs: this grid must not complete before its upstream does)

    if (warp == 4) {
        // ---------------- producer ----------------
        // no griddepcontrol.wait here: the cross K/V cache is written once before the decode loop starts, so when this kernel is
        // launched as a programmatic dependent the first K chunks are already in flight while the upstream GEMM drains
        if (lane == 0) {
            const uint8_t* kb = reinterpret_cast<const uint8_t*>(kcross + (long long)kvh * Tlen * 64);
            const uint8_t* vb = reinterpret_cast<const uint8_t*>(vcross + (long long)kvh * Tlen * 64);
            for (int c = 0; c < 2 * chunks; ++c) {
                const int stage = c % kCrossStages;
                const uint32_t ph = (c / kCrossStages) & 1;
                mbar_wait(&empty_bar[stage], ph ^ 1);
                mbar_expect_tx(&full_bar[stage], kCrossStageBytes);
                const uint8_t* src = c < chunks ? kb + (long long)c * kCrossStageBytes : vb + (long long)(c - chunks) * kCrossStageBytes;
                bulk_load_1d(ring + stage * kCrossStageBytes, src, kCrossStageBytes, &full_bar[stage]);
            }
        }
        return;
    }
    // ---------------- consumers (128 threads) ----------------
    pdl_wait();                      // the q partials come from the upstream GEMM
    if (tid < 64) {
        float q = bq[h * 64 + tid];
        for (int s = 0; s < splits; ++s) q += partial[((long long)s * Bp + b) * dm + h * 64 + tid];
        sq[tid] = q * 0.125f;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    const int sub = lane & 7;        // 16-byte piece of the 128-byte row: dims sub*8 .. sub*8+7
    const int rsel = lane >> 3;      // row within a group of 4
    float qv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) qv[j] = sq[sub * 8 + j];

    // K phase: scores[t] = q . K[t]
    for (int c = 0; c < chunks; ++c) {
        const int stage = c % kCrossStages;
        const uint32_t ph = (c / kCrossStages) & 1;
        mbar_wait(&full_bar[stage], ph);
        const uint8_t* tile = ring + stage * kCrossStageBytes;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = warp * 4 + rsel + 16 * i;
            float acc = 0.f;
            if (r < kCrossRows) {
                const uint4 u = *reinterpret_cast<const uint4*>(tile + r * 128 + sub * 16);
                const float2 a0 = T16<T>::unpack2(u.x), a1 = T16<T>::unpack2(u.y), a2 = T16<T>::unpack2(u.z), a3 = T16<T>::unpack2(u.w);
                acc = qv[0] * a0.x + qv[1] * a0.y + qv[2] * a1.x + qv[3] * a1.y + qv[4] * a2.x + qv[5] * a2.y + qv[6] * a3.x + qv[7] * a3.y;
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            acc += __shfl_xor_sync(0xffffffffu, acc, 2);
            acc += __shfl_xor_sync(0xffffffffu, acc, 4);
            if (sub == 0 && r < kCrossRows) scores[c * kCrossRows + r] = acc;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    // softmax over Tlen scores (consumers only)
    float mx = -INFINITY;
    for (int t = tid; t < Tlen; t += 128) mx = fmaxf(mx, scores[t]);
    mx = warp_max(mx);
    if (lane == 0) red[warp] = mx;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    float sm = 0.f;
    for (int t = tid; t < Tlen; t += 128) {
        const float p = __expf(scores[t] - mx);
        scores[t] = p;
        sm += p;
    }
    sm = warp_sum(sm);
    asm volatile("bar.sync 1, 128;" ::: "memory");   // everyone has read red[] (max) before it is reused
    if (lane == 0) red[warp] = sm;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    const float inv = 1.f / (red[0] + red[1] + red[2] + red[3]);
    if (align_scratch != nullptr && ((align_mask >> h) & 1u)) {
        // alignment head: export the normalised softmax row (word timestamps); slot = rank of h among the layer's alignment heads
        const int slot = __popc(align_mask & ((1u << h) - 1u));
        float* dst = align_scratch + ((long long)slot * B + b) * Tlen;
        for (int t = tid; t < Tlen; t += 128) dst[t] = scores[t] * inv;
    }

    // V phase: out[d] = sum_t p[t] V[t][d]
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int c = chunks; c < 2 * chunks; ++c) {
        const int stage = c % kCrossStages;
        const uint32_t ph = (c / kCrossStages) & 1;
        mbar_wait(&full_bar[stage], ph);
        const uint8_t* tile = ring + stage * kCrossStageBytes;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = warp * 4 + rsel + 16 * i;
            if (r < kCrossRows) {
                const float p = scores[(c - chunks) * kCrossRows + r];
                const uint4 u = *reinterpret_cast<const uint4*>(tile + r * 128 + sub * 16);
                const float2 a0 = T16<T>::unpack2(u.x), a1 = T16<T>::unpack2(u.y), a2 = T16<T>::unpack2(u.z), a3 = T16<T>::unpack2(u.w);
                acc[0] += p * a0.x; acc[1] += p * a0.y; acc[2] += p * a1.x; acc[3] += p * a1.y;
                acc[4] += p * a2.x; acc[5] += p * a2.y; acc[6] += p * a3.x; acc[7] += p * a3.y;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");   // red[] (sum) consumed by everyone
    if (rsel == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[warp * 64 + sub * 8 + j] = acc[j];
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (tid < 64) {
        const float o = (red[tid] + red[64 + tid] + red[128 + tid] + red[192 + tid]) * inv;
        out[(long long)b * dm + h * 64 + tid] = T16<T>::from_f(o);
    }
}

static size_t cross_smem_bytes(int T) {
    return (size_t)kCrossStages * kCrossStageBytes + (size_t)((T + 3) & ~3) * 4 + 64 * 4 + (4 * 64 + 32) * 4 + 2 * kCrossStages * 8 + 64;
}

// The beam-search form (NQ rows share one K/V block) lives in cross_attention_mq.cu: both products on the tensor cores.

__global__ void decoder_align_mean_kernel(const float* __restrict__ scratch, int n_slots, const int32_t* __restrict__ steps,
                                          const int32_t* __restrict__ done, __half* __restrict__ out, int B, int Tlen, int max_rows) {
    const int b = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
    // launched after the sampler advanced the row's step: steps[b] = tokenIndex + 1 = the row of this step's slice; a window whose
    // segment just completed (or completed earlier) gets no row - the reference breaks out of its loop before updateAlignmentWeights
    // (TextDecoder.swift:668-674,709-717)
    // (row 0 is never a step's row: steps[b] is still 0 only after a language-detection pre-step, which has no alignment row)
    const int row = steps[b];
    if (t >= Tlen || row < 1 || row >= max_rows || done[b]) return;
    float a = 0.f;
    for (int s = 0; s < n_slots; ++s) a += scratch[((long long)s * B + b) * Tlen + t];   // fixed order: deterministic
    out[((long long)b * max_rows + row) * Tlen + t] = __float2half(a / (float)n_slots);
}

wk_status decoder_align_mean(const float* scratch, int n_slots, const int32_t* steps, const int32_t* done, void* out_f16, int B, int T,
                             int max_rows, cudaStream_t stream) {
    launch_k(decoder_align_mean_kernel, dim3((T + 255) / 256, B), dim3(256), 0, stream, 0, scratch, n_slots, steps, done, (__half*)out_f16, B, T, max_rows);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_align_mean launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

wk_status decoder_cross_attention(const float* partial, int splits, int Bp, const float* bq, const void* kcross,
                                  const void* vcross, void* out, int B, int H, int T, int dtype, cudaStream_t stream,
                                  const int32_t* done, float* align_scratch, uint32_t align_mask, int kv_div) {
    if (kv_div < 1 || B % kv_div != 0) { set_error("decoder_cross_attention: %d rows do not split into groups of %d", B, kv_div); return WK_ERR_INVALID_ARGUMENT; }
    if (T % kCrossRows != 0) { set_error("decoder_cross_attention: n_audio_ctx %d not a multiple of %d", T, kCrossRows); return WK_ERR_INVALID_ARGUMENT; }
    if (kv_div > 1 && kv_div <= 8 && align_scratch == nullptr)   // beam search: one CTA per (window, head) serves all beams from one K/V pass
        return decoder_cross_attention_mq(partial, splits, Bp, bq, kcross, vcross, out, B, H, T, dtype, stream, done, kv_div);
    const size_t smem = cross_smem_bytes(T);
    static bool attr_set[2] = {false, false};
    const int ti = dtype == WK_DTYPE_F16 ? 1 : 0;
    if (!attr_set[ti]) {
        cudaError_t e = dtype == WK_DTYPE_F16
            ? cudaFuncSetAttribute(decoder_cross_attention_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)
            : cudaFuncSetAttribute(decoder_cross_attention_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(cross): %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
        attr_set[ti] = true;
    }
    if (dtype == WK_DTYPE_F16)
        launch_k(decoder_cross_attention_kernel<__half>, dim3(B * H), dim3(kCrossThreads), smem, stream, 4, partial, splits, Bp, bq, (const __half*)kcross, (const __half*)vcross, (__half*)out, B, H, T, done, align_scratch, align_mask, kv_div);
    else
        launch_k(decoder_cross_attention_kernel<__nv_bfloat16>, dim3(B * H), dim3(kCrossThreads), smem, stream, 4, partial, splits, Bp, bq, (const __nv_bfloat16*)kcross, (const __nv_bfloat16*)vcross, (__nv_bfloat16*)out, B, H, T, done, align_scratch, align_mask, kv_div);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("decoder_cross_attention launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

// =====================================================================================================
// K7: fused logits filters + greedy sampler + decode-loop state update.  One CTA per sequence; the logits row
// (V f32, 207 KB for V = 51866) is staged once in shared memory, masks are applied while it streams in, and the
// max / log-sum-exp / argmax reductions of TimestampRulesFilter and GreedyTokenSampler run out of smem.
// =====================================================================================================
static constexpr int kSamplerThreads = 1024;

struct ArgMax { float v; int i; };
__device__ __forceinline__ ArgMax argmax_better(ArgMax a, ArgMax b) {
    // larger value wins; ties -> lower index (first maximal index, like argmax)
    if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
    return a;
}

__global__ void __launch_bounds__(kSamplerThreads)
sampler_kernel(const float* __restrict__ logits, long long ld_logits, SamplerParams p, DecodeState st,
               const int32_t* __restrict__ tokens_in, int ld_tokens, const int32_t* __restrict__ n_tokens_in,
               int32_t* __restrict__ token_out, float* __restrict__ logprob_out, float* __restrict__ filtered_out) {
    extern __shared__ __align__(16) float srow[];  // [V]
    __shared__ float scratch[32];
    __shared__ int sflag[8];     // 0: ts filter active, 1: lo0, 2: hi0 (interval A), 3: lo1, 4: hi1 (interval B), 5: blank active
    __shared__ ArgMax sarg[32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int V = p.vocab;
    const bool loop_mode = p.loop_mode != 0;
    pdl_launch_dependents();
    pdl_wait();
    if (loop_mode && st.done[b]) return;   // ended window: its logits row is not even read
    // per-row options: the decode loop reads them from the row's RowParams, the stateless entry from the call
    RowParams R;
    if (loop_mode) {
        R = st.rp[b];
    } else {
        R.prompt_len = -1; R.sample_begin_ts = p.sample_begin_ts; R.sample_begin_blank = p.sample_begin_blank; R.max_steps = 0;
        R.temperature = p.temperature; R.top_k = p.top_k; R.has_first_thr = 0; R.first_thr = 0.f; R.seed = p.seed;
        R.suppress_off = 0; R.n_suppress = p.n_suppress;
    }
    const int32_t* toks = loop_mode ? st.tokens + b * kMaxCtx : tokens_in + (long long)b * ld_tokens;
    const int n_tok = loop_mode ? st.n_tokens[b] : n_tokens_in[b];
    const wk_special_tokens& S = p.st;
    // DecodingOptions.detectLanguage (TranscribeTask.swift:339-365, TextDecoder.swift:420-539): a detecting row's first pass runs SOT at
    // position 0, so its logits are detectLanguage's.  Pass 0 samples the language from them (LanguageLogitsFilter, then the rung's
    // sampler; no other filter); pass 1 is the ordinary step.  A pre-step (prompt not starting with SOT) runs pass 0 only.  The branch is
    // per row: rows that do not detect run pass 1 alone.
    const bool detect = loop_mode && R.lang_flags != 0 && st.steps[b] == 0 && st.lang_tok[b] < 0;
    const bool prestep = detect && (R.lang_flags & kLangPreStep) != 0;
    for (int pass = detect ? 0 : 1; pass < (prestep ? 1 : 2); ++pass) {
    const bool lang_pass = pass == 0;
    if (tid == 0) {
        // ---- TimestampRulesFilter rule state (LogitsFilter.swift:72-109)
        int active = 0, loA = 0, hiA = 0, loB = 0, hiB = 0;
        if (!lang_pass && R.sample_begin_ts >= 0) {
            int sb = -1;
            if (p.is_multilingual) {
                const int lim = n_tok < 3 ? n_tok : 3;
                for (int i = 0; i < lim; ++i)
                    if (toks[i] == S.transcribe_token || toks[i] == S.translate_token) { sb = max(i + 1, R.sample_begin_ts); break; }
            } else {
                sb = R.sample_begin_ts;
            }
            if (sb >= 0 && sb <= n_tok) {
                active = 1;
                if (n_tok > sb) {
                    const int ns = n_tok - sb;
                    const bool last_ts = ns >= 1 && toks[n_tok - 1] >= S.time_token_begin;
                    const bool pen_ts = ns < 2 || toks[n_tok - 2] >= S.time_token_begin;
                    if (last_ts) {
                        if (pen_ts) { loA = S.time_token_begin; hiA = V; }   // has to be non-timestamp
                        else { loA = 0; hiA = S.end_token; }                 // cannot be normal text
                    }
                    int last_time = -1;
                    for (int i = n_tok - 1; i >= sb; --i)
                        if (toks[i] >= S.time_token_begin) { last_time = toks[i]; break; }
                    if (last_time >= 0) {
                        const int ts_last = (last_ts && !pen_ts) ? last_time : last_time + 1;
                        loB = S.time_token_begin; hiB = ts_last;
                    }
                }
            }
        }
        sflag[0] = active; sflag[1] = loA; sflag[2] = hiA; sflag[3] = loB; sflag[4] = hiB;
        sflag[5] = (!lang_pass && R.sample_begin_blank >= 0 && n_tok == R.sample_begin_blank) ? 1 : 0;   // SuppressBlankFilter
        sflag[6] = (lang_pass || (!loop_mode && p.language_tokens != nullptr && n_tok >= p.language_sample_begin)) ? 1 : 0;  // LanguageLogitsFilter
    }
    __syncthreads();
    const int ts_active = sflag[0], loA = sflag[1], hiA = sflag[2], loB = sflag[3], hiB = sflag[4];
    const int blank_active = sflag[5], lang_active = sflag[6];
    const float* row = logits + (long long)b * ld_logits;

    // ---- stream the row into smem with the interval / single-token masks applied
    for (int i = tid; i < V; i += kSamplerThreads) {
        float x = lang_active ? -INFINITY : row[i];
        if (blank_active && (i == S.whitespace_token || i == S.end_token)) x = -INFINITY;
        if (ts_active) {
            if (i == S.no_timestamps_token) x = -INFINITY;
            if ((i >= loA && i < hiA) || (i >= loB && i < hiB)) x = -INFINITY;
        }
        srow[i] = x;
    }
    __syncthreads();
    if (lang_active) {
        for (int j = tid; j < p.n_language_tokens; j += kSamplerThreads) {
            const int t = p.language_tokens[j];
            if (t >= 0 && t < V) srow[t] = row[t];
        }
        __syncthreads();
        // re-apply the filters that run after a (custom-positioned) language filter
        for (int j = tid; j < p.n_language_tokens; j += kSamplerThreads) {
            const int i = p.language_tokens[j];
            if (i < 0 || i >= V) continue;
            if (blank_active && (i == S.whitespace_token || i == S.end_token)) srow[i] = -INFINITY;
            if (ts_active && (i == S.no_timestamps_token || (i >= loA && i < hiA) || (i >= loB && i < hiB))) srow[i] = -INFINITY;
        }
        __syncthreads();
    }
    for (int j = tid; j < (lang_pass ? 0 : R.n_suppress); j += kSamplerThreads) {   // SuppressTokensFilter
        const int t = p.suppress[R.suppress_off + j];
        if (t >= 0 && t < V) srow[t] = -INFINITY;
    }
    __syncthreads();

    // ---- reductions: max over text / timestamp partitions
    const int tsb = (ts_active && S.time_token_begin > 0 && S.time_token_begin < V) ? S.time_token_begin : V;
    float mtext = -INFINITY, mts = -INFINITY;
    for (int i = tid; i < V; i += kSamplerThreads) {
        const float x = srow[i];
        if (i < tsb) mtext = fmaxf(mtext, x); else mts = fmaxf(mts, x);
    }
    mtext = block_max(mtext, scratch);
    mts = block_max(mts, scratch);
    const float mall = fmaxf(mtext, mts);
    float sall = 0.f, sts = 0.f;
    for (int i = tid; i < V; i += kSamplerThreads) {
        const float x = srow[i];
        if (x == -INFINITY) continue;
        sall += __expf(x - mall);
        if (i >= tsb) sts += __expf(x - mts);
    }
    sall = block_sum(sall, scratch);
    sts = block_sum(sts, scratch);
    float lse = mall + logf(sall);
    // "sum of probability over timestamps is above any other token" (LogitsFilter.swift:124-127,144-242)
    bool ts_wins = false;
    if (tsb < V && mts > -INFINITY) {
        const float lse_ts = mts + logf(sts);
        const float ts_logprob = lse_ts - lse;
        const float max_text_logprob = mtext - lse;
        ts_wins = ts_logprob > max_text_logprob;
        if (ts_wins) lse = lse_ts;
    }
    const int lo = ts_wins ? tsb : 0;
    if (ts_wins && filtered_out) {
        for (int i = tid; i < tsb; i += kSamplerThreads) srow[i] = -INFINITY;
        __syncthreads();
    }
    if (filtered_out) {
        for (int i = tid; i < V; i += kSamplerThreads) filtered_out[(long long)b * V + i] = srow[i];
        __syncthreads();
    }
    // ---- block-wide argmax (first maximal index) over [lo, V); srow is only read
    auto block_argmax = [&]() -> ArgMax {
        ArgMax best = {-INFINITY, 0x7fffffff};
        for (int i = lo + tid; i < V; i += kSamplerThreads) {
            const float x = srow[i];
            if (x > best.v) { best.v = x; best.i = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ArgMax other;
            other.v = __shfl_xor_sync(0xffffffffu, best.v, o);
            other.i = __shfl_xor_sync(0xffffffffu, best.i, o);
            best = argmax_better(best, other);
        }
        __syncthreads();
        if ((tid & 31) == 0) sarg[tid >> 5] = best;
        __syncthreads();
        best = sarg[tid & 31];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ArgMax other;
            other.v = __shfl_xor_sync(0xffffffffu, best.v, o);
            other.i = __shfl_xor_sync(0xffffffffu, best.i, o);
            best = argmax_better(best, other);
        }
        return best;   // identical in every thread
    };
    if (loop_mode && !lang_pass && p.beam.beam > 1) {
        // beam search: rank the row's (beam + 1) best tokens of the filtered log-softmax, best first (whisper BeamSearchDecoder.update step 1);
        // the per-window merge and every state update happen in beam_update_kernel
        const int k = p.beam.beam + 1;
        for (int kk = 0; kk < k; ++kk) {
            const ArgMax a = block_argmax();
            const bool ok = a.v != -INFINITY && a.i >= 0 && a.i < V;   // (a NaN row yields the initial index: no candidate)
            if (tid == 0) {
                p.beam.cand_tok[b * (kMaxBeam + 1) + kk] = ok ? a.i : -1;
                p.beam.cand_lp[b * (kMaxBeam + 1) + kk] = ok ? a.v - lse : -INFINITY;
                if (ok) srow[a.i] = -INFINITY;
            }
            __syncthreads();
        }
        return;
    }
    ArgMax best;
    float lp_sampled = 0.f;
    if (R.temperature == 0.f) {
        best = block_argmax();
        lp_sampled = best.v - lse;
    } else {
        // GreedyTokenSampler with temperature (TokenSampler.swift:57-73 / :140-180): logits / T, softmax over the whole
        // (filtered) vocabulary, top-k, multinomial draw inside the top-k mass, logprob = log softmax prob of the draw.
        // The reference draws with Float.random (non-deterministic); here the draw is Philox(seed, row, step).  The language draw uses
        // subsequence 2^32 + row, which no token draw of any row reaches.
        const float inv_t = 1.f / R.temperature;
        const float zmax = (ts_wins ? mts : mall) * inv_t;
        float z = 0.f;
        for (int i = lo + tid; i < V; i += kSamplerThreads) {
            const float x = srow[i];
            if (x != -INFINITY) z += __expf(x * inv_t - zmax);
        }
        z = block_sum(z, scratch);
        __shared__ float topv[32];
        __shared__ int topi[32];
        const int k = R.top_k < 1 ? 1 : (R.top_k > 32 ? 32 : R.top_k);
        int kk = 0;
        for (; kk < k; ++kk) {
            const ArgMax a = block_argmax();
            if (a.v == -INFINITY) break;
            if (tid == 0) { topv[kk] = __expf(a.v * inv_t - zmax) / z; topi[kk] = a.i; srow[a.i] = -INFINITY; }
            __syncthreads();
        }
        __syncthreads();
        float mass = 0.f;
        for (int j = 0; j < kk; ++j) mass += topv[j];
        curandStatePhilox4_32_10_t rng;
        if (lang_pass) curand_init(R.seed, (1ull << 32) + (unsigned long long)b, 0ull, &rng);
        else curand_init(R.seed, (unsigned long long)b, (unsigned long long)(loop_mode ? st.steps[b] : n_tok), &rng);
        const float u = 1.f - curand_uniform(&rng);   // [0, 1)
        const float rnd = u * mass;
        float acc = 0.f;
        int chosen = kk > 0 ? kk - 1 : 0;
        for (int j = 0; j < kk; ++j) {
            acc += topv[j];
            if (rnd < acc) { chosen = j; break; }
        }
        best.i = kk > 0 ? topi[chosen] : 0x7fffffff;
        best.v = 0.f;
        lp_sampled = kk > 0 ? logf(topv[chosen]) : -INFINITY;
    }
    if (tid == 0) {
        int tok = best.i;
        float lp = lp_sampled;
        // a row with no finite logit (every token masked, or a NaN from upstream) has no argmax: end the window there and flag it instead
        // of feeding an out-of-range id to the next embedding lookup (the host reports WhisperError.decodingLogitsFailed for the window)
        const bool bad = tok < 0 || tok >= V;
        sflag[7] = lang_pass && bad;
        if (lang_pass) {
            // the detected language; the embed kernel forces it at the prompt's language position
            if (bad) { st.error[b] = 1; st.done[b] = 1; }
            else {
                st.lang_tok[b] = tok; st.lang_lp[b] = lp;
                if (R.lang_slot >= 0) st.tokens[b * kMaxCtx + R.lang_slot] = tok;
            }
        } else {
        if (bad) { tok = S.end_token; lp = -INFINITY; }
        if (token_out) token_out[b] = bad ? -1 : tok;
        if (logprob_out) logprob_out[b] = lp;
        if (loop_mode) {
            // decodeText bookkeeping (TextDecoder.swift:654-686)
            const int step = st.steps[b];
            const bool first_low = (step == 0) && R.has_first_thr && (lp < R.first_thr);
            const bool completed = (tok == S.end_token) || (n_tok >= p.max_ctx - 1) || first_low;
            st.next_token[b] = tok;
            st.steps[b] = step + 1;
            if (bad) st.error[b] = 1;
            if (completed) {
                st.done[b] = 1;
                st.first_low[b] = first_low ? 1 : 0;
            } else {
                if (!(step < R.prompt_len - 1)) {   // !isPrefill
                    st.tokens[b * kMaxCtx + n_tok] = tok;
                    st.logprobs[b * kMaxCtx + n_tok] = lp;
                    st.n_tokens[b] = n_tok + 1;
                }
                if (step + 1 >= R.max_steps) st.done[b] = 1;   // loop bound min(sampleLength, 223) reached (TextDecoder.swift:566)
            }
        }
        }
    }
    if (lang_pass) {   // (uniform over the CTA) pass 1 restages srow; a row without a finite language logit ends here
        __syncthreads();
        if (sflag[7]) return;
    }
    }
}

// =====================================================================================================
// Beam search step (oracle/beam_ref.py is the specification).  One CTA per window; rows r0 .. r0 + beam - 1 are its beams.
// =====================================================================================================
static constexpr int kBeamThreads = 128;

__global__ void __launch_bounds__(kBeamThreads)
beam_update_kernel(DecodeState st, BeamState bs, wk_special_tokens S, int max_ctx) {
    __shared__ int32_t s_tok[kMaxBeam][kMaxCtx];
    __shared__ float s_lp[kMaxBeam][kMaxCtx];
    __shared__ int32_t s_anc[kMaxBeam][kMaxCtx];
    __shared__ float c_score[kMaxBeam * (kMaxBeam + 1)], c_lp[kMaxBeam * (kMaxBeam + 1)];
    __shared__ int c_src[kMaxBeam * (kMaxBeam + 1)], c_tok[kMaxBeam * (kMaxBeam + 1)], c_ord[kMaxBeam * (kMaxBeam + 1)];
    __shared__ int n_src[kMaxBeam], n_tokv[kMaxBeam];
    __shared__ float n_lp[kMaxBeam], n_score[kMaxBeam];
    __shared__ int f_src[kMaxCand]; __shared__ float f_score[kMaxCand];
    __shared__ int sh[4];   // 0: mode (0 prefill/plain advance, 1 ranked, 2 ended without ranking)  1: new finished count  2: window done  3: finished before
    const int g = blockIdx.x, tid = threadIdx.x, beam = bs.beam, r0 = g * beam;
    pdl_launch_dependents();
    pdl_wait();
    if (st.done[r0]) return;
    const RowParams R = st.rp[r0];
    const int step = st.steps[r0], n_tok = st.n_tokens[r0], P = R.prompt_len;
    const int C1 = kMaxBeam + 1;
    if (tid == 0) {
        const int gtok = bs.cand_tok[r0 * C1];
        const float glp = bs.cand_lp[r0 * C1];
        const bool bad = gtok < 0;
        const bool first_low = (step == 0) && R.has_first_thr && (glp < R.first_thr);
        int mode = 0, done = 0;
        int nf_before = bs.n_fin[g];
        int nf_new = 0;
        if (bad) { done = 1; mode = 2; }
        else if (step < P - 1) {                       // prefill: every beam is the same forced copy; greedy bookkeeping
            if (gtok == S.end_token || first_low) done = 1;
        } else if (n_tok >= max_ctx - 1 || first_low) {
            done = 1; mode = 2;
        } else {
            mode = 1;
            const int considered = (step == P - 1) ? 1 : beam;   // identical beams count once
            int nc = 0;
            for (int j = 0; j < considered; ++j)
                for (int k = 0; k <= beam; ++k) {
                    const int t = bs.cand_tok[(r0 + j) * C1 + k];
                    if (t < 0) continue;
                    const float v = bs.cand_lp[(r0 + j) * C1 + k];
                    c_score[nc] = bs.sum_lp[r0 + j] + v; c_lp[nc] = v; c_src[nc] = j; c_tok[nc] = t; c_ord[nc] = nc; ++nc;
                }
            for (int i = 1; i < nc; ++i) {             // stable insertion sort, best score first
                const int o = c_ord[i];
                int k = i - 1;
                while (k >= 0 && c_score[c_ord[k]] < c_score[o]) { c_ord[k + 1] = c_ord[k]; --k; }
                c_ord[k + 1] = o;
            }
            int saved = 0;
            for (int i = 0; i < nc && saved < beam; ++i) {
                const int o = c_ord[i];
                if (c_tok[o] == S.end_token) {
                    if (nf_before + nf_new < bs.max_candidates) { f_src[nf_new] = c_src[o]; f_score[nf_new] = c_score[o]; ++nf_new; }
                } else {
                    n_src[saved] = c_src[o]; n_tokv[saved] = c_tok[o]; n_lp[saved] = c_lp[o]; n_score[saved] = c_score[o]; ++saved;
                }
            }
            for (; saved < beam; ++saved) {            // (cannot happen with beam + 1 candidates per beam; keeps the state well formed)
                n_src[saved] = n_src[saved > 0 ? saved - 1 : 0]; n_tokv[saved] = n_tokv[saved > 0 ? saved - 1 : 0]; n_lp[saved] = 0.f; n_score[saved] = -INFINITY;
            }
            if (nf_before + nf_new >= bs.max_candidates) done = 1;
        }
        if (!done && step + 1 >= R.max_steps) done = 1;   // loop bound (TextDecoder.swift:566)
        sh[0] = mode; sh[1] = nf_new; sh[2] = done; sh[3] = nf_before;
        for (int j = 0; j < beam; ++j) {
            const int r = r0 + j;
            st.steps[r] = step + 1;
            if (bad) st.error[r] = 1;
            if (mode != 1) st.next_token[r] = bad ? S.end_token : gtok;
            if (done) { st.done[r] = 1; st.first_low[r] = first_low ? 1 : 0; }
            bs.anc[r * kMaxCtx + step] = r;             // position `step` of this row's cache was written by the row itself
        }
    }
    __syncthreads();
    if (sh[0] != 1) return;
    // ---- ranked step: histories and ancestry move to the surviving beams
    for (int i = tid; i < beam * kMaxCtx; i += kBeamThreads) {
        const int j = i / kMaxCtx, t = i % kMaxCtx;
        s_tok[j][t] = st.tokens[(r0 + j) * kMaxCtx + t];
        s_lp[j][t] = st.logprobs[(r0 + j) * kMaxCtx + t];
        s_anc[j][t] = bs.anc[(r0 + j) * kMaxCtx + t];
    }
    __syncthreads();
    for (int f = 0; f < sh[1]; ++f) {                   // newly finished: prefix of the source beam + EOT (log-prob 0, like sampler.finalize)
        const int slot = g * kMaxCand + sh[3] + f, src = f_src[f];
        for (int t = tid; t < n_tok; t += kBeamThreads) {
            bs.fin_tokens[slot * kMaxCtx + t] = s_tok[src][t];
            bs.fin_lps[slot * kMaxCtx + t] = s_lp[src][t];
        }
        if (tid == 0) {
            bs.fin_tokens[slot * kMaxCtx + n_tok] = S.end_token;
            bs.fin_lps[slot * kMaxCtx + n_tok] = 0.f;
            bs.fin_len[slot] = n_tok + 1;
            bs.fin_score[slot] = f_score[f];
        }
    }
    if (tid == 0) bs.n_fin[g] = sh[3] + sh[1];
    for (int i = tid; i < beam * kMaxCtx; i += kBeamThreads) {
        const int j = i / kMaxCtx, t = i % kMaxCtx, r = r0 + j, src = n_src[j];
        if (t < n_tok) { st.tokens[r * kMaxCtx + t] = s_tok[src][t]; st.logprobs[r * kMaxCtx + t] = s_lp[src][t]; }
        else if (t == n_tok) { st.tokens[r * kMaxCtx + t] = n_tokv[j]; st.logprobs[r * kMaxCtx + t] = n_lp[j]; }
        if (t <= step) bs.anc[r * kMaxCtx + t] = (t == step) ? r0 + src : s_anc[src][t];
    }
    if (tid < beam) {
        const int r = r0 + tid;
        st.n_tokens[r] = n_tok + 1;
        st.next_token[r] = n_tokv[tid];
        bs.sum_lp[r] = n_score[tid];
    }
}

wk_status beam_update(DecodeState st, BeamState beam, wk_special_tokens sp, int max_ctx, int groups, cudaStream_t stream) {
    if (beam.beam < 2 || beam.beam > kMaxBeam || beam.max_candidates < 1 || beam.max_candidates > kMaxCand) {
        set_error("beam_update: beam %d / candidates %d outside [2, %d] / [1, %d]", beam.beam, beam.max_candidates, kMaxBeam, kMaxCand);
        return WK_ERR_INVALID_ARGUMENT;
    }
    launch_k(beam_update_kernel, dim3(groups), dim3(kBeamThreads), 0, stream, 8, st, beam, sp, max_ctx);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("beam_update launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

wk_status sampler_filter_sample(const float* logits, int64_t ld_logits, SamplerParams p, DecodeState st, const int32_t* tokens,
                                int ld_tokens, const int32_t* n_tokens, int32_t* token_out, float* logprob_out,
                                float* filtered_out, int B, cudaStream_t stream) {
    const size_t smem = (size_t)p.vocab * sizeof(float);
    if (smem > 220 * 1024) { set_error("sampler: vocab %d too large for the shared-memory row", p.vocab); return WK_ERR_INVALID_ARGUMENT; }
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(sampler_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(sampler): %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
        attr_set = true;
    }
    launch_k(sampler_kernel, dim3(B), dim3(kSamplerThreads), smem, stream, 8, logits, (long long)ld_logits, p, st, tokens, ld_tokens,
             n_tokens, token_out, logprob_out, filtered_out);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("sampler launch: %s", cudaGetErrorString(e)); return WK_ERR_CUDA; }
    return WK_OK;
}

}  // namespace wk
