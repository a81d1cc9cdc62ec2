// msm_pair.cuh — batched-affine pre-accumulation of the sorted MSM entry list.
//
// The bucket accumulation of msm.cuh adds points one by one into an XYZZ accumulator (G1: 9.5 modmul-equivalents per
// entry, G2: 27.5).  In affine coordinates an addition costs 2M + 1S plus one field inversion; with Montgomery's
// simultaneous-inversion trick the inversion is shared by thousands of independent additions (3 more multiplies each).
// Such additions exist in the sorted list: neighbours with equal keys belong to the same bucket.  One round adds list
// positions (2j, 2j+1) when their keys are equal and passes both through otherwise, so key order is preserved and every
// bucket roughly halves:
//
//   k_pair_prefix   slot j = k*T + t of thread t: classify the pair, write the prefix product of the thread's earlier
//                   denominators to pre[j] and the output count (1 or 2) of the slot; the thread's product to tprod[t].
//                   Round 0 reads the points through the sorted values (table index | sign << 31); that gather needs only
//                   the x coordinates here.  Later rounds read the previous round's output stream.
//   cub scan        exclusive sum of the output counts = output positions (no bucket offsets)
//   k_pair_invert   one warp per PAIR_THREADS thread products: shuffle scans, ONE field inversion, the inverse of every
//                   thread's product back to invp[t].  Each lane of a warp inverts, so no CTA waits on one warp.
//   k_pair_apply    back-substitution from the thread's last slot to its first, the affine sums to dst[pos[j]].
//
// Rounds run while the list averages more than PAIR_STOP_DENSITY entries per bucket (msm.cuh msm_buckets); what remains
// goes through the unchanged segmented XYZZ accumulation / fold / reduce of msm.cuh with vals == nullptr.
//
// Special cases inside a pair (pair_kind; tests/test_gpu_batch_affine.py, tests/host/host_batch_affine_check.cpp):
// either point at infinity ((0,0), reference build/snarkjs.js:6068-6086), P + P (doubling: denominator 2y, numerator
// 3x^2), P + (-P) (the sum is (0,0) and stays in the list as a point at infinity).
#pragma once
#include "ec.cuh"

namespace sb {

enum { PAIR_COPY = 0, PAIR_ADD = 1, PAIR_DBL = 2, PAIR_INF = 3, PAIR_TAKE2 = 4 };

// What the sum of two points of one bucket needs (y1, y2 carry their signs).  ADD and DBL go through the shared inversion
// of `den`; INF is P + (-P); TAKE2 / COPY: the first / second operand is the point at infinity, the sum is the other one.
template <class F> SB_HD int pair_kind(const F& x1, const F& y1, const F& x2, const F& y2, F& den) {
    den = F::one();
    if (x1.is_zero() & y1.is_zero()) return PAIR_TAKE2;
    if (x2.is_zero() & y2.is_zero()) return PAIR_COPY;
    if (x1 == x2) {
        if ((y1 == y2) & !y1.is_zero()) { den = F::dbl(y1); return PAIR_DBL; }
        return PAIR_INF;
    }
    den = F::sub(x2, x1);
    return PAIR_ADD;
}
// The sum of the pair; inv = 1 / den for ADD and DBL (unused otherwise).
template <class F> SB_HD Affine<F> pair_sum(int kind, const F& x1, const F& y1, const F& x2, const F& y2, const F& inv) {
    Affine<F> r;
    if (kind == PAIR_ADD || kind == PAIR_DBL) {
        F lam;
        if (kind == PAIR_ADD) lam = F::mul_i(F::sub(y2, y1), inv);
        else { F xx = F::sqr_i(x1); lam = F::mul_i(F::add(F::dbl(xx), xx), inv); }
        r.x = F::sub(F::sub(F::sqr_i(lam), x1), x2);
        r.y = F::sub(F::mul_i(lam, F::sub(x1, r.x)), y1);
    } else if (kind == PAIR_INF) { r.x = F::zero(); r.y = F::zero(); }
    else if (kind == PAIR_TAKE2) { r.x = x2; r.y = y2; }
    else { r.x = x1; r.y = y1; }
    return r;
}

#ifdef __CUDACC__
static constexpr int PAIR_THREADS = 128;                     // CTA size of the round kernels = thread products per inversion
static constexpr int PAIR_LANE_PRODUCTS = PAIR_THREADS / 32;  // thread products per lane in k_pair_invert

// point s of a round's input list; round 0 (FIRST) reads it through the sorted value (index | sign << 31)
template <class F, bool FIRST>
__device__ __forceinline__ uint64_t pair_index(const uint32_t* __restrict__ vals, uint64_t s, bool& neg) {
    if (FIRST) { const uint32_t v = vals[s]; neg = (v >> 31) != 0; return v & 0x7fffffffu; }
    neg = false; return s;
}
template <class F, bool FIRST>
__device__ __forceinline__ void pair_load(const Affine<F>* __restrict__ pts, const uint32_t* __restrict__ vals, uint64_t s, F& x, F& y) {
    bool neg; const uint64_t i = pair_index<F, FIRST>(vals, s, neg);
    load_affine<F>(pts + i, 0, x, y);
    y = F::cneg(y, neg);
}

template <class F, int MODE> __device__ __forceinline__ F shfl_f(const F& v, int d) {   // MODE 0: up, 1: down, 2: index
    constexpr int NW = sizeof(F) / 4;
    union U { F f; uint32_t w[NW]; __device__ U() {} };
    U a, r; a.f = v;
#pragma unroll
    for (int k = 0; k < NW; k++)
        r.w[k] = MODE == 0 ? __shfl_up_sync(0xffffffffu, a.w[k], d) : MODE == 1 ? __shfl_down_sync(0xffffffffu, a.w[k], d) : __shfl_sync(0xffffffffu, a.w[k], d);
    return r.f;
}

// counts: the round's input (counts[0] = list length n).  Slots j <= Jub get their output count (0 past the list).
template <class F, bool FIRST>
__global__ void __launch_bounds__(PAIR_THREADS)
k_pair_prefix(const Affine<F>* __restrict__ src, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ keys,
              const uint64_t* __restrict__ counts, uint64_t Jub, uint32_t K, F* __restrict__ pre, F* __restrict__ tprod,
              uint32_t* __restrict__ outc) {
    const uint64_t n = counts[0], J = (n + 1) / 2;
    const uint64_t T = (uint64_t)gridDim.x * blockDim.x, t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    F acc = F::one();
    for (uint32_t k = 0; k < K; k++) {
        const uint64_t j = k * T + t;
        if (j > Jub) break;
        uint32_t c = 0;
        if (j < J) {
            const uint64_t s = 2 * j;
            c = 1;
            if (s + 1 < n) {
                if (keys[s] != keys[s + 1]) c = 2;
                else {
                    // only the x coordinates, unless a special case needs the y coordinates (same result as pair_kind)
                    bool n1, n2;
                    const uint64_t i1 = pair_index<F, FIRST>(vals, s, n1), i2 = pair_index<F, FIRST>(vals, s + 1, n2);
                    const F x1 = load_vec(&src[i1].x), x2 = load_vec(&src[i2].x);
                    F den; int kind = PAIR_ADD;
                    if (x1.is_zero() | x2.is_zero() | (x1 == x2))
                        kind = pair_kind<F>(x1, F::cneg(load_vec(&src[i1].y), n1), x2, F::cneg(load_vec(&src[i2].y), n2), den);
                    else den = F::sub(x2, x1);
                    if (kind == PAIR_ADD || kind == PAIR_DBL) { store_vec(pre + j, acc); acc = F::mul_i(acc, den); }
                }
            }
        }
        outc[j] = c;
    }
    store_vec(tprod + t, acc);
}

// One warp per PAIR_THREADS consecutive thread products (T is a multiple of PAIR_THREADS): invp[t] = 1 / tprod[t].
// Thread 0 also writes the next round's counts from the scanned output positions (pos[Jub] = list length).
template <class F>
__global__ void __launch_bounds__(128)
k_pair_invert(const F* __restrict__ tprod, uint64_t T, F* __restrict__ invp, const uint32_t* __restrict__ pos, uint64_t Jub,
              uint64_t* __restrict__ counts_out, uint64_t wave) {
    const uint64_t gid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (gid == 0) msm_fill_counts(counts_out, pos[Jub], MSM_SEG, MSM_SEG / 2, wave);
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t w = gid >> 5;
    if (w * PAIR_THREADS >= T) return;                        // the whole warp leaves together
    const F* p = tprod + w * PAIR_THREADS + lane * PAIR_LANE_PRODUCTS;
    F q[PAIR_LANE_PRODUCTS], l = F::one();
#pragma unroll
    for (int i = 0; i < PAIR_LANE_PRODUCTS; i++) { q[i] = l; l = F::mul_i(l, load_vec(p + i)); }
    F inc = l, suf = l;                                       // inclusive prefix / suffix products of the lane products
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) {
        F a = shfl_f<F, 0>(inc, d), b = shfl_f<F, 1>(suf, d);
        if (lane >= (uint32_t)d) inc = F::mul_i(a, inc);
        if (lane + d < 32) suf = F::mul_i(suf, b);
    }
    const F total = shfl_f<F, 2>(inc, 31);
    F before = shfl_f<F, 0>(inc, 1), after = shfl_f<F, 1>(suf, 1);
    if (lane == 0) before = F::one();
    if (lane == 31) after = F::one();
    F r = F::mul_i(F::mul_i(PairInvF(total), before), after);    // 1 / (this lane's product)
    F* o = invp + w * PAIR_THREADS + lane * PAIR_LANE_PRODUCTS;
#pragma unroll
    for (int i = PAIR_LANE_PRODUCTS - 1; i >= 0; i--) {
        store_vec(o + i, F::mul_i(r, q[i]));
        if (i) r = F::mul_i(r, load_vec(p + i));
    }
}

template <class F, bool FIRST>
__global__ void __launch_bounds__(PAIR_THREADS)
k_pair_apply(const Affine<F>* __restrict__ src, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ keys,
             const uint64_t* __restrict__ counts, uint32_t K, const F* __restrict__ pre, const F* __restrict__ invp,
             const uint32_t* __restrict__ pos, Affine<F>* __restrict__ dst, uint32_t* __restrict__ dst_keys) {
    const uint64_t n = counts[0], J = (n + 1) / 2;
    const uint64_t T = (uint64_t)gridDim.x * blockDim.x, t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    F running = load_vec(invp + t);                           // 1 / (product of the thread's denominators so far)
    for (int k = (int)K - 1; k >= 0; k--) {
        const uint64_t j = (uint64_t)k * T + t;
        if (j >= J) continue;
        const uint64_t s = 2 * j;
        const uint32_t o = pos[j], key = keys[s];
        Affine<F> a, b;
        pair_load<F, FIRST>(src, vals, s, a.x, a.y);
        if (s + 1 < n) {
            pair_load<F, FIRST>(src, vals, s + 1, b.x, b.y);
            const uint32_t key2 = keys[s + 1];
            if (key2 != key) { store_vec(dst + o + 1, b); dst_keys[o + 1] = key2; }
            else {
                F den;
                const int kind = pair_kind<F>(a.x, a.y, b.x, b.y, den);
                F inv = den;
                if (kind == PAIR_ADD || kind == PAIR_DBL) { inv = F::mul_i(running, load_vec(pre + j)); running = F::mul_i(running, den); }
                a = pair_sum<F>(kind, a.x, a.y, b.x, b.y, inv);
            }
        }
        store_vec(dst + o, a); dst_keys[o] = key;
    }
}
#endif  // __CUDACC__

}  // namespace sb
