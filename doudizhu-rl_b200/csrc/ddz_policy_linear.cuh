// ddz_policy_linear.cuh -- a linear policy head evaluated only at the legal ids: logit(b, id) = W[id] . h_b + bias[id],
// computed straight from the hidden vector h_b, then sampled, scored and differentiated by the bodies of the fixed-head
// kernels (ddz_policy.cuh), so that nothing of size [B, 13551] is ever made.  One warp per env, as there; the weight and
// bias gradients are sums over the entries of each id, taken over the CSR entries sorted by id (the caller's stable sort)
// in fixed-length chunks whose partials are added in chunk order: no floating-point atomics, the same bits every call.
// The kernels live in their own namespace, apart from the environment's and the dense head's kernels.
#pragma once
#include "ddz_policy.cuh"

namespace ddz {
namespace linear_head {

using policy_head::EnvList;
using policy_head::env_list;
using policy_head::kFull;
using policy_head::kWarps;

constexpr int kMaxHidden = 1024;        // largest H
constexpr int kChunk = 128;             // entries of the sorted order per weight-gradient chunk (a fixed constant: the
                                        // chunk boundaries, hence the order of every sum, depend on the inputs alone)

// 16 bytes of DT = kVec<DT> elements; bfloat16 is widened exactly
template <int DT>
constexpr int kVec = DT == DDZ_DTYPE_F32 ? 4 : 8;

template <int DT>
DDZ_DEV void widen(const uint4& q, float* f) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if constexpr (DT == DDZ_DTYPE_F32) {
            f[k] = __uint_as_float(w[k]);
        } else {
            f[2 * k] = __uint_as_float(w[k] << 16);
            f[2 * k + 1] = __uint_as_float(w[k] & 0xFFFF0000u);
        }
    }
}
template <int DT>
DDZ_DEV uint4 narrow(const float* f) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if constexpr (DT == DDZ_DTYPE_F32) w[k] = __float_as_uint(f[k]);
        else w[k] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f[2 * k])) |
                    ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f[2 * k + 1])) << 16);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}
template <int DT>
DDZ_DEV void store_scalar(void* p, size_t i, float v) {
    if constexpr (DT == DDZ_DTYPE_F32) reinterpret_cast<float*>(p)[i] = v;
    else reinterpret_cast<uint16_t*>(p)[i] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
}

// The head: hidden rows of H elements at hidden + b * ld, weight [DDZ_NUM_ACTION_IDS][H], bias [DDZ_NUM_ACTION_IDS] or
// NULL; one dtype.  Row pointers are 16-byte aligned (checked by the launchers).
template <int DT>
struct Head {
    const void* hidden;
    const void* weight;
    const void* bias;
    int H;
    long long ld;

    DDZ_DEV const uint4* hidden_row(long long b) const {
        return reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(hidden) + (size_t)b * (size_t)ld * (16 / kVec<DT>));
    }
    DDZ_DEV const uint4* weight_row(int id) const {
        return reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(weight) + (size_t)id * (size_t)H * (16 / kVec<DT>));
    }

    // THE logit of action id `id` for env b (the whole warp; every lane returns the same float): lane k sums the products
    // of the 16-byte pieces k, k + 32, ... of W[id] and h_b, piece by piece and element by element in increasing order
    // (fmaf), the lanes' sums are added by the xor butterfly 16, 8, 4, 2, 1, then bias[id] is added.  The order depends on
    // H alone, never on B or the launch.  A negative id (not a move) gives -inf, as the dense gather does.
    DDZ_DEV float logit(int b, int id, int lane) const {
        if (id < 0) return -CUDART_INF_F;
        const uint4* x = hidden_row(b);
        const uint4* wr = weight_row(id);
        const int nq = H / kVec<DT>;
        float acc = 0.f;
#pragma unroll 2
        for (int q = lane; q < nq; q += 32) {
            float a[kVec<DT>], c[kVec<DT>];
            widen<DT>(__ldg(wr + q), a);
            widen<DT>(__ldg(x + q), c);
#pragma unroll
            for (int k = 0; k < kVec<DT>; k++) acc = fmaf(a[k], c[k], acc);
        }
        acc = policy_head::warp_sum(acc);
        return bias ? acc + policy_head::load_logit<DT>(bias, (size_t)id) : acc;
    }

    // the logit source of the fixed-head bodies (policy_head::DenseLogits' interface): ids and logits of env b's n entries
    // into shared memory; the largest logit (NaN ignored) is folded lane by lane in DenseLogits' order, so that the same
    // logits give the same m bit for bit
    DDZ_DEV float gather(const uint64_t* actions, long long lo, int n, int b, int16_t* ids, float* l, int lane,
                         bool& any_nan) const {
        for (int i = lane; i < n; i += 32) ids[i] = (int16_t)move_id(actions[lo + i]);
        __syncwarp();
        float m = -CUDART_INF_F;
        bool nan = false;
        for (int i = 0; i < n; i++) {
            const float v = logit(b, ids[i], lane);
            if ((i & 31) == lane) {
                l[i] = v;
                m = fmaxf(m, v);
                nan |= v != v;
            }
        }
        __syncwarp();
        any_nan = __any_sync(kFull, nan);
        return policy_head::warp_max(m);
    }
};

// the stored entries of env b's list (all of them unless the capacity cut the list)
DDZ_DEV long long stored_entries(const int32_t* offsets, long long cap, int b) {
    return max(0ll, min((long long)offsets[b + 1], cap) - (long long)offsets[b]);
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_logits(const int32_t* __restrict__ offsets,
                                                               const uint64_t* __restrict__ actions, long long cap,
                                                               Head<DT> hd, float* __restrict__ out, int64_t* stats, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float slog[kWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    const EnvList e = env_list(offsets, cap, b);
    if (e.n < 0) {                                         // cut or dropped: NaN at the stored entries, counted once
        const long long stored = stored_entries(offsets, cap, b);
        for (long long i = lane; i < stored; i += 32) out[e.lo + i] = CUDART_NAN_F;
        if (lane == 0 && stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
        return;
    }
    bool nan;
    hd.gather(actions, e.lo, e.n, b, sids[w], slog[w], lane, nan);
    for (int i = lane; i < e.n; i += 32) out[e.lo + i] = slog[w][i];
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_sample(const int32_t* __restrict__ offsets,
                                                               const uint64_t* __restrict__ actions, long long cap,
                                                               Head<DT> hd, float T, uint64_t seed, uint64_t env0,
                                                               uint32_t stepno, const uint8_t* __restrict__ env_mask,
                                                               uint32_t* meta, int32_t* choice, int32_t* ids_out,
                                                               float* logp_out, float* entropy_out, int64_t* stats, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float slog[kWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    policy_head::sample_env(hd, b, lane, offsets, actions, cap, T, seed, env0, stepno, env_mask, meta, choice, ids_out,
                            logp_out, entropy_out, stats, sids[w], slog[w]);
}

template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_logprob(const int32_t* __restrict__ offsets,
                                                                const uint64_t* __restrict__ actions, long long cap,
                                                                Head<DT> hd, const int32_t* __restrict__ chosen,
                                                                float* logp_out, float* entropy_out, float* lse_out,
                                                                int64_t* stats, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float slog[kWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    policy_head::logprob_env(hd, b, lane, offsets, actions, cap, chosen, logp_out, entropy_out, lse_out, stats, sids[w],
                             slog[w]);
}

// The per-env part of the gradient: grad_legal at the env's stored entries (the values the dense backward puts at the
// legal ids; 0 for an empty, cut or dropped list) and grad_hidden[b] = sum_i grad_legal_i W[id_i], each 16-byte piece
// summed by one lane in list order (fmaf).
template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_backward(const int32_t* __restrict__ offsets,
                                                                 const uint64_t* __restrict__ actions, long long cap,
                                                                 Head<DT> hd, const int32_t* __restrict__ chosen,
                                                                 const float* __restrict__ lse_in,
                                                                 const float* __restrict__ grad_logp,
                                                                 const float* __restrict__ grad_entropy,
                                                                 float* __restrict__ grad_legal, void* __restrict__ grad_hidden,
                                                                 long long ld_g, int B) {
    __shared__ int16_t sids[kWarps][DDZ_MAX_LEGAL];
    __shared__ float sg[kWarps][DDZ_MAX_LEGAL];
    constexpr int V = kVec<DT>;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kWarps + w;
    if (b >= B) return;
    const int16_t* ids = sids[w];
    const float* g = sg[w];
    const int n = policy_head::grad_env(hd, b, lane, offsets, actions, cap, chosen, lse_in, grad_logp, grad_entropy, sids[w],
                                        sg[w]);
    const long long lo = offsets[b], stored = stored_entries(offsets, cap, b);
    for (long long i = lane; i < stored; i += 32) grad_legal[lo + i] = i < n ? g[i] : 0.f;
    uint4* row = reinterpret_cast<uint4*>(reinterpret_cast<char*>(grad_hidden) + (size_t)b * (size_t)ld_g * (16 / V));
    for (int q = lane; q < hd.H / V; q += 32) {
        float acc[V];
#pragma unroll
        for (int k = 0; k < V; k++) acc[k] = 0.f;
#pragma unroll 4
        for (int i = 0; i < n; i++) {
            const int id = ids[i];
            if (id >= 0) {
                float wv[V];
                widen<DT>(__ldg(hd.weight_row(id) + q), wv);
#pragma unroll
                for (int k = 0; k < V; k++) acc[k] = fmaf(g[i], wv[k], acc[k]);
            }
        }
        row[q] = narrow<DT>(acc);
    }
}

// Weight and bias gradients, pass 1.  The sorted entries are cut into chunks of kChunk positions of `order`; one warp per
// chunk.  Within a chunk the positions form runs of one id; a run's partial sum (grad_legal[e] * h[env(e)], and
// grad_legal[e] for the bias) is taken in position order, i.e. env order.  A run that holds its id's whole segment is the
// id's gradient and is stored as its row; otherwise the partial goes to the chunk's workspace slot 0 (the id's segment
// began in an earlier chunk) or 1 (it begins here and goes on), and k_linear_grad_combine adds it up.
template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_grad_chunks(const int32_t* __restrict__ offsets, int B, long long n,
                                                                    Head<DT> hd, const float* __restrict__ grad_legal,
                                                                    const int32_t* __restrict__ order,
                                                                    const int32_t* __restrict__ id_offsets,
                                                                    void* __restrict__ grad_weight, void* __restrict__ grad_bias,
                                                                    float* __restrict__ ws) {
    __shared__ int senv[kWarps][kChunk];
    __shared__ float sgl[kWarps][kChunk];
    __shared__ int16_t sid[kWarps][kChunk];
    constexpr int V = kVec<DT>;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long k = (long long)blockIdx.x * kWarps + w, p0 = k * kChunk;
    if (p0 >= n) return;
    const int cnt = (int)min((long long)kChunk, n - p0);
    for (int j = lane; j < cnt; j += 32) {
        const long long p = p0 + j;
        int lo = 0, hi = DDZ_NUM_ACTION_IDS;               // the id of position p: the last x with id_offsets[x] <= p
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (id_offsets[mid] <= p) lo = mid; else hi = mid - 1;
        }
        const int e = order[p];
        int bl = 0, bh = B - 1;                            // the env of entry e: the last b with offsets[b] <= e
        while (bl < bh) {
            const int mid = (bl + bh + 1) >> 1;
            if (offsets[mid] <= e) bl = mid; else bh = mid - 1;
        }
        sid[w][j] = (int16_t)(lo < DDZ_NUM_ACTION_IDS ? lo : -1);     // past the last segment: no id, not counted
        senv[w][j] = bl;
        sgl[w][j] = grad_legal[e];
    }
    __syncwarp();
    const int16_t* ids = sid[w];
    const int* env = senv[w];
    const float* gl = sgl[w];
    const size_t stride = (size_t)hd.H + 4;                // floats per workspace slot: H, then the bias
    float* slot0 = ws + (size_t)(2 * k) * stride;
    // where the run of id x that ends at this chunk's position j goes: its row (0), slot 0 or slot 1 (the returned pointer)
    auto target = [&](int x) -> float* {
        const long long s = id_offsets[x], e = id_offsets[x + 1];
        if (s >= p0 && e <= p0 + cnt) return nullptr;
        return s < p0 ? slot0 : slot0 + stride;
    };
    for (int q = lane; q < hd.H / V; q += 32) {
        float acc[V];
#pragma unroll
        for (int t = 0; t < V; t++) acc[t] = 0.f;
        for (int j0 = 0; j0 < cnt; j0 += 4) {
            uint4 hv[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int j = j0 + u;
                hv[u] = j < cnt && ids[j] >= 0 ? __ldg(hd.hidden_row(env[j]) + q) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int j = j0 + u;
                if (j >= cnt) break;
                const int x = ids[j];
                if (x < 0) continue;
                float hf[V];
                widen<DT>(hv[u], hf);
#pragma unroll
                for (int t = 0; t < V; t++) acc[t] = fmaf(gl[j], hf[t], acc[t]);
                if (j + 1 == cnt || ids[j + 1] != x) {
                    float* dst = target(x);
                    if (dst) {
#pragma unroll
                        for (int t = 0; t < V; t += 4)
                            *reinterpret_cast<float4*>(dst + (size_t)q * V + t) = make_float4(acc[t], acc[t + 1], acc[t + 2], acc[t + 3]);
                    } else {
                        reinterpret_cast<uint4*>(reinterpret_cast<char*>(grad_weight) + (size_t)x * hd.H * (16 / V))[q] =
                            narrow<DT>(acc);
                    }
#pragma unroll
                    for (int t = 0; t < V; t++) acc[t] = 0.f;
                }
            }
        }
    }
    if (grad_bias && lane == 0) {
        float acc = 0.f;
        for (int j = 0; j < cnt; j++) {
            const int x = ids[j];
            if (x < 0) break;                              // the positions without an id come last
            acc += gl[j];
            if (j + 1 == cnt || ids[j + 1] != x) {
                float* dst = target(x);
                if (dst) dst[hd.H] = acc;
                else store_scalar<DT>(grad_bias, (size_t)x, acc);
                acc = 0.f;
            }
        }
    }
}

// acc[0 .. V) += the V floats at p (16-byte aligned)
template <int V>
DDZ_DEV void add_floats(const float* p, float* acc) {
#pragma unroll
    for (int t = 0; t < V; t += 4) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p + t));
        acc[t] += v.x;
        acc[t + 1] += v.y;
        acc[t + 2] += v.z;
        acc[t + 3] += v.w;
    }
}

// Pass 2, one warp per id: an id with no entry gets an exact-zero row (and bias); an id whose segment spans chunks adds its
// partials in chunk order, slot 1 of its first chunk, then slot 0 of each later one.  The other ids were written by pass 1.
template <int DT>
__global__ void __launch_bounds__(kWarps * 32) k_linear_grad_combine(int H, const int32_t* __restrict__ id_offsets,
                                                                     void* __restrict__ grad_weight,
                                                                     void* __restrict__ grad_bias,
                                                                     const float* __restrict__ ws) {
    constexpr int V = kVec<DT>;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int x = blockIdx.x * kWarps + w;
    if (x >= DDZ_NUM_ACTION_IDS) return;
    const long long s = id_offsets ? id_offsets[x] : 0, e = id_offsets ? id_offsets[x + 1] : 0;
    const long long k0 = s / kChunk, k1 = (e - 1) / kChunk;
    if (e > s && k0 == k1) return;
    const size_t stride = (size_t)H + 4;
    const float* first = ws + (size_t)(2 * k0 + 1) * stride;     // read only when e > s
    for (int q = lane; q < H / V; q += 32) {
        float acc[V];
#pragma unroll
        for (int t = 0; t < V; t++) acc[t] = 0.f;
        if (e > s) {
            add_floats<V>(first + (size_t)q * V, acc);
#pragma unroll 8
            for (long long c = k0 + 1; c <= k1; c++) add_floats<V>(ws + (size_t)(2 * c) * stride + (size_t)q * V, acc);
        }
        reinterpret_cast<uint4*>(reinterpret_cast<char*>(grad_weight) + (size_t)x * H * (16 / V))[q] = narrow<DT>(acc);
    }
    if (grad_bias && lane == 0) {
        float acc = 0.f;
        if (e > s) {
            acc += first[H];
            for (long long c = k0 + 1; c <= k1; c++) acc += ws[(size_t)(2 * c) * stride + H];
        }
        store_scalar<DT>(grad_bias, (size_t)x, acc);
    }
}

}  // namespace linear_head
}  // namespace ddz
