// ddz_policy.cuh -- fixed-head policies over the action ids: a softmax over the 13 551-entry output head restricted to the
// legal ids of every env, without a dense mask.  One warp per env: the lanes turn the env's list into ids (move_id, in
// increasing order), gather logits[b * ld + id] into shared memory, and reduce.  Sampling, log-probability, entropy and
// the gradient of the last two all read only the N legal logits of an env (mean 5.6, at most DDZ_MAX_LEGAL).
// The kernels live in their own namespace, apart from the environment's kernels.
#pragma once
#include <cuda_bf16.h>
#include "ddz_ids.cuh"

namespace ddz {
namespace policy_head {

constexpr int kWarps = 8;
constexpr unsigned kFull = 0xFFFFFFFFu;

template <int DT>
DDZ_DEV float load_logit(const void* p, size_t i) {
    if constexpr (DT == DDZ_DTYPE_F32) return reinterpret_cast<const float*>(p)[i];
    return __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(p)[i] << 16);
}

DDZ_DEV float warp_max(float v) {
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
DDZ_DEV float warp_sum(float v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
// inclusive scan across the lanes (Hillis-Steele: step d adds the value of lane - d), the order the header pins for the draw
DDZ_DEV float lane_scan(float v, int lane) {
    for (int d = 1; d < 32; d <<= 1) {
        const float t = __shfl_up_sync(kFull, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// The stored part of env b's list: n entries from lo, or n = -1 when the list was cut or dropped by the capacity (the
// stored part is not the whole list) or is longer than DDZ_MAX_LEGAL.
struct EnvList { long long lo; int n; };
DDZ_DEV EnvList env_list(const int32_t* offsets, long long cap, int b) {
    const long long lo = offsets[b], full = max(0ll, (long long)offsets[b + 1] - lo);
    const long long stored = max(0ll, min(full, cap - lo));
    return {lo, (stored < full || full > DDZ_MAX_LEGAL) ? -1 : (int)full};
}

// ids and logits of the n entries into shared memory; returns the largest logit (NaN ignored; -inf for none) and sets
// any_nan when a logit is NaN.
template <int DT>
DDZ_DEV float gather_logits(const uint64_t* actions, long long lo, int n, const void* logits, size_t row, int16_t* ids,
                            float* l, int lane, bool& any_nan) {
    float m = -CUDART_INF_F;
    bool nan = false;
    for (int i = lane; i < n; i += 32) {
        const int id = move_id(actions[lo + i]);
        const float v = id >= 0 ? load_logit<DT>(logits, row + (size_t)id) : -CUDART_INF_F;
        ids[i] = (int16_t)id;
        l[i] = v;
        m = fmaxf(m, v);
        nan |= v != v;
    }
    __syncwarp();
    any_nan = __any_sync(kFull, nan);
    return warp_max(m);
}

// One pass over the entries with z = (l - m) / T, w = exp(z), their running sums as the header pins them (32-entry
// chunks in list order, each scanned across the lanes and added to the running sum at lane 31 of the chunk before).
// Returns S = the running sum at the LAST entry with w > 0 -- not the one at lane 31 of the last chunk, whose different
// association over the zero padding can round above it -- or NaN when no entry has w > 0; and sum_wz = sum of w * z
// over the entries with w > 0 (any order).
DDZ_DEV float weight_pass(const float* l, int n, float m, float T, int lane, float& sum_wz) {
    float carry = 0.f, wz = 0.f, S = CUDART_NAN_F;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const float z = i < n ? (l[i] - m) / T : -CUDART_INF_F;
        const float w = i < n ? expf(z) : 0.f;
        if (w > 0.f) wz += w * z;
        const float run = carry + lane_scan(w, lane);
        const unsigned pos = __ballot_sync(kFull, w > 0.f);
        if (pos) S = __shfl_sync(kFull, run, 31 - __clz(pos));
        carry = __shfl_sync(kFull, run, 31);
    }
    sum_wz = warp_sum(wz);
    return S;
}

// (NaN first, then larger value, then lower index): torch.argmax's order
DDZ_DEV bool argmax_before(float va, int ia, float vb, int ib) {
    const bool na = va != va, nb = vb != vb;
    if (na != nb) return na;
    if (!na && va != vb) return va > vb;
    return ia < ib;
}

// The legal logits of a dense head: logits[b * ld + id].  A logit source gathers the ids and logits of env b's n entries
// into shared memory as gather_logits does; the bodies below take any source, so that a head which computes its legal
// logits (ddz_policy_linear.cuh) samples, scores and differentiates with the same float32 arithmetic as the dense one.
template <int DT>
struct DenseLogits {
    const void* logits;
    long long ld;
    DDZ_DEV float gather(const uint64_t* actions, long long lo, int n, int b, int16_t* ids, float* l, int lane,
                         bool& any_nan) const {
        return gather_logits<DT>(actions, lo, n, logits, (size_t)b * (size_t)ld, ids, l, lane, any_nan);
    }
};

// ddz_policy_sample of env b (one warp; ids / l: the warp's DDZ_MAX_LEGAL entries of shared memory)
template <class Src>
DDZ_DEV void sample_env(const Src& src, int b, int lane, const int32_t* __restrict__ offsets,
                        const uint64_t* __restrict__ actions, long long cap, float T, uint64_t seed, uint64_t env0,
                        uint32_t stepno, const uint8_t* __restrict__ env_mask, uint32_t* meta, int32_t* choice,
                        int32_t* ids_out, float* logp_out, float* entropy_out, int64_t* stats, int16_t* ids, float* l) {
    int c = -1;
    float lp = 0.f, h = 0.f;
    bool cut = false, bad = false;
    const bool live = (env_mask == nullptr || env_mask[b] != 0) && offsets[b + 1] > offsets[b];
    if (live) {
        const EnvList e = env_list(offsets, cap, b);
        cut = e.n < 0;
        if (!cut) {
            bool nan;
            const float m = src.gather(actions, e.lo, e.n, b, ids, l, lane, nan);
            const float Te = T > 0.f ? T : 1.f;
            // no draw without a finite positive total: all legal logits -inf, or (T > 0) a NaN or +inf among them
            bad = (m == -CUDART_INF_F && !nan) || (T > 0.f && (nan || m == CUDART_INF_F));
            if (!bad) {
                float wz = 0.f;
                const float S = nan ? CUDART_NAN_F : weight_pass(l, e.n, m, Te, lane, wz);
                if (T > 0.f) {
                    const float u = (float)(philox(seed, env0 + (uint64_t)b, stepno) >> 8) * (1.0f / 16777216.0f);
                    const float target = u * S;
                    // only entries with w > 0 take part; u * S < S, so the last of them (whose running sum is S) always
                    // qualifies and a list with a finite positive S always gets an entry of non-zero probability
                    float carry = 0.f;
                    for (int base = 0; base < e.n && c < 0; base += 32) {
                        const int i = base + lane;
                        const float wi = i < e.n ? expf((l[i] - m) / Te) : 0.f;
                        const float run = carry + lane_scan(wi, lane);
                        const unsigned hit = __ballot_sync(kFull, wi > 0.f && run > target);
                        if (hit) c = base + __ffs(hit) - 1;
                        carry = __shfl_sync(kFull, run, 31);
                    }
                } else {
                    float bv = -CUDART_INF_F;
                    int bi = INT_MAX;
                    for (int i = lane; i < e.n; i += 32)
                        if (argmax_before(l[i], i, bv, bi)) { bv = l[i]; bi = i; }
                    for (int o = 16; o > 0; o >>= 1) {
                        const float ov = __shfl_xor_sync(kFull, bv, o);
                        const int oi = __shfl_xor_sync(kFull, bi, o);
                        if (argmax_before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
                    }
                    c = bi;
                }
                if (c >= 0) {
                    const float logS = logf(S);
                    lp = (l[c] - m) / Te - logS;
                    h = logS - wz / S;
                }
            }
        }
    }
    if (lane == 0) {
        if (cut || bad) {
            c = -1;
            lp = h = 0.f;
            if (stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
            if (bad && meta) meta[b] |= 0x20u;                 // sticky error; a cut list is the capacity's, not the env's
        }
        choice[b] = c;
        ids_out[b] = c >= 0 ? (int)ids[c] : -1;
        logp_out[b] = lp;
        entropy_out[b] = h;
    }
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_policy_sample(const int32_t* __restrict__ offsets,
                                                               const uint64_t* __restrict__ actions, long long cap,
                                                               const void* __restrict__ logits, long long ld, float T,
                                                               uint64_t seed, uint64_t env0, uint32_t stepno,
                                                               const uint8_t* __restrict__ env_mask, uint32_t* meta,
                                                               int32_t* choice, int32_t* ids_out, float* logp_out,
                                                               float* entropy_out, int64_t* stats, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float slog[kWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    sample_env(DenseLogits<DT>{logits, ld}, b, lane, offsets, actions, cap, T, seed, env0, stepno, env_mask, meta, choice,
               ids_out, logp_out, entropy_out, stats, sids[w], slog[w]);
}

// Training forward of env b: log-probability of the chosen ids[b] and entropy under the legal-restricted softmax (T = 1),
// and the log-sum-exp over the legal set for the backward.
template <class Src>
DDZ_DEV void logprob_env(const Src& src, int b, int lane, const int32_t* __restrict__ offsets,
                         const uint64_t* __restrict__ actions, long long cap, const int32_t* __restrict__ chosen,
                         float* logp_out, float* entropy_out, float* lse_out, int64_t* stats, int16_t* ids, float* l) {
    const EnvList e = env_list(offsets, cap, b);
    float lp = 0.f, h = 0.f, lse = -CUDART_INF_F;
    bool count = false;
    if (e.n < 0) {
        lp = h = lse = CUDART_NAN_F;
        count = true;
    } else if (e.n > 0) {
        bool nan;
        const float m = src.gather(actions, e.lo, e.n, b, ids, l, lane, nan);
        float wz = 0.f;
        const float S = nan ? CUDART_NAN_F : weight_pass(l, e.n, m, 1.f, lane, wz);
        const float logS = logf(S);
        const int want = chosen[b];
        int c = -1;
        for (int base = 0; base < e.n && c < 0; base += 32) {
            const unsigned hit = __ballot_sync(kFull, base + lane < e.n && ids[base + lane] == want);
            if (hit) c = base + __ffs(hit) - 1;
        }
        lse = m + logS;
        h = logS - wz / S;
        lp = c >= 0 ? (l[c] - m) - logS : -CUDART_INF_F;
        count = c < 0 || S != S;                           // an id off the list, or no softmax (S = NaN): counted once
    }
    if (lane == 0) {
        if (count && stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
        logp_out[b] = lp;
        entropy_out[b] = h;
        if (lse_out) lse_out[b] = lse;
    }
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_policy_logprob(const int32_t* __restrict__ offsets,
                                                                const uint64_t* __restrict__ actions, long long cap,
                                                                const void* __restrict__ logits, long long ld,
                                                                const int32_t* __restrict__ chosen, float* logp_out,
                                                                float* entropy_out, float* lse_out, int64_t* stats, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float slog[kWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    logprob_env(DenseLogits<DT>{logits, ld}, b, lane, offsets, actions, cap, chosen, logp_out, entropy_out, lse_out, stats,
                sids[w], slog[w]);
}

// The gradient of env b at its legal entries, g_lp (1[id = chosen] - p) - g_ent p (log p + H), into g[0 .. n) with the
// ids in ids[0 .. n); returns n (0 for an empty, cut or dropped list).
template <class Src>
DDZ_DEV int grad_env(const Src& src, int b, int lane, const int32_t* __restrict__ offsets,
                     const uint64_t* __restrict__ actions, long long cap, const int32_t* __restrict__ chosen,
                     const float* __restrict__ lse_in, const float* __restrict__ grad_logp,
                     const float* __restrict__ grad_entropy, int16_t* ids, float* g) {
    const EnvList e = env_list(offsets, cap, b);
    const int n = max(e.n, 0);                             // a cut or dropped list gets a zero gradient
    if (n > 0) {
        bool nan;
        src.gather(actions, e.lo, n, b, ids, g, lane, nan);
        const float lse = lse_in[b];
        const float glp = grad_logp ? grad_logp[b] : 0.f, gent = grad_entropy ? grad_entropy[b] : 0.f;
        float plp = 0.f;                                   // H = -sum p log p
        for (int i = lane; i < n; i += 32) {
            const float lq = g[i] - lse, p = expf(lq);
            if (p > 0.f) plp += p * lq;
        }
        const float H = -warp_sum(plp);
        const int want = chosen[b];
        for (int i = lane; i < n; i += 32) {
            const float lq = g[i] - lse, p = expf(lq);
            float v = glp * ((ids[i] == want ? 1.f : 0.f) - p);
            if (p > 0.f) v -= gent * p * (lq + H);
            g[i] = v;
        }
        __syncwarp();
    }
    return n;
}

// The gradient row of env b over all 13 551 ids, written once: g_lp (1[id = chosen] - p) - g_ent p (log p + H) on the
// legal ids, 0 elsewhere.  The warp first turns the list into (id, gradient) pairs in shared memory, then every lane stores
// 16-byte pieces lane, lane + 32, ... of the row (coalesced), finding the ids of each piece by a merge walk that only moves
// forward -- k_legal_mask's row writer.  The elements before the first 16-byte boundary and after the last one are
// stored singly.
template <int DT>
DDZ_DEV void store_elem(void* row, int k, float v) {
    if constexpr (DT == DDZ_DTYPE_F32) reinterpret_cast<float*>(row)[k] = v;
    else reinterpret_cast<uint16_t*>(row)[k] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
DDZ_DEV int find_id(const int16_t* ids, int n, int id) {
    int lo = 0, hi = n;                                    // first entry >= id
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ids[mid] < id) lo = mid + 1; else hi = mid; }
    return lo < n && ids[lo] == id ? lo : -1;
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_policy_logprob_backward(const int32_t* __restrict__ offsets,
                                                                         const uint64_t* __restrict__ actions, long long cap,
                                                                         const void* __restrict__ logits, long long ld,
                                                                         const int32_t* __restrict__ chosen,
                                                                         const float* __restrict__ lse_in,
                                                                         const float* __restrict__ grad_logp,
                                                                         const float* __restrict__ grad_entropy,
                                                                         void* grad, long long grad_ld, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float sg[kWarps][DDZ_MAX_LEGAL];
    constexpr int kEsz = DT == DDZ_DTYPE_F32 ? 4 : 2, kSpan = 16 / kEsz;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    int16_t* ids = sids[w];
    float* g = sg[w];
    const int n = grad_env(DenseLogits<DT>{logits, ld}, b, lane, offsets, actions, cap, chosen, lse_in, grad_logp,
                           grad_entropy, ids, g);
    char* row = reinterpret_cast<char*>(grad) + (size_t)b * (size_t)grad_ld * kEsz;
    const int head = (int)(((0u - (uint32_t)reinterpret_cast<uintptr_t>(row)) & 15u) / kEsz);   // elements before a boundary
    const int nmid = (DDZ_NUM_ACTION_IDS - head) / kSpan, tail = head + kSpan * nmid;
    if (lane < head) { const int k = find_id(ids, n, lane); store_elem<DT>(row, lane, k >= 0 ? g[k] : 0.f); }
    if (lane >= 16 && tail + lane - 16 < DDZ_NUM_ACTION_IDS) {
        const int id = tail + lane - 16, k = find_id(ids, n, id);
        store_elem<DT>(row, id, k >= 0 ? g[k] : 0.f);
    }
    uint4* mid = reinterpret_cast<uint4*>(row + (size_t)head * kEsz);
    int p = 0;
    for (int c = lane; c < nmid; c += 32) {
        const int base = head + c * kSpan;
        float v[kSpan];
#pragma unroll
        for (int k = 0; k < kSpan; k++) v[k] = 0.f;
        while (p < n && ids[p] < base) p++;
        for (; p < n && ids[p] < base + kSpan; p++) {
            const int d = ids[p] - base;
#pragma unroll
            for (int k = 0; k < kSpan; k++) if (d == k) v[k] = g[p];
        }
        uint32_t q[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if constexpr (DT == DDZ_DTYPE_F32) q[k] = __float_as_uint(v[k]);
            else q[k] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v[2 * k])) |
                        ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v[2 * k + 1])) << 16);
        }
        mid[c] = make_uint4(q[0], q[1], q[2], q[3]);
    }
}

}  // namespace policy_head
}  // namespace ddz
