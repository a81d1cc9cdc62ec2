// msm.cuh — Pippenger multi-scalar multiplication on one B200 (templated on the coordinate field).
//
// Replaces ffjavascript engine_multiexp (_multiExp/_multiExpChunk, reference build/snarkjs.js:14517-14669)
// and wasmcurves build_multiexp (g?m_multiexpAffine_chunk 5542-5695, _getChunk 5471-5540,
// _reduceTable 5819-5907).  The reference runs one task per (point-chunk, window), each re-copying its
// chunk; here all windows are processed in one pass over the scalars:
//
//   k_digits      scalars -> signed c-bit digits; one (key = window*B + |d|-1, val = index | sign<<31)
//                 entry per non-zero digit   (B = 2^(c-1) buckets per window)
//   radix sort    entries by key (cub::DeviceRadixSort, library plumbing)
//   k_accumulate  balanced segmented bucket accumulation: every thread owns SEG consecutive sorted
//                 entries regardless of bucket sizes (robust to witness-like skew: many 0/1 scalars),
//                 gathers affine bases with 128-bit loads, XYZZ mixed adds; a run that starts inside
//                 the segment is written straight to its bucket, the thread's first run goes to a
//                 "head" partial that the next (32x smaller) level folds in.
//   k_fold        same segmented walk over the head partials (full XYZZ adds) until one thread is left
//   k_reduce      per window sum_b (b+1)*bucket[b] by chunked running sums + small scalar multiply,
//                 then a shared-memory tree to one point per window
//   host          Horner over the W window sums (W*c doublings on 1 point: latency-bound, CPU is faster)
#pragma once
#include <algorithm>
#include <cuda_runtime.h>
#include "ec.cuh"
#include "msm_geom.h"

namespace sb {

static constexpr int MSM_SEG = 32;          // sorted entries per thread in k_accumulate / k_fold
static constexpr int MSM_ACC_THREADS = 128;
static constexpr int MSM_RED_CHUNK = 16;    // buckets per thread in k_reduce
static constexpr uint32_t MSM_INVALID_KEY = 0xffffffffu;
static constexpr int MSM_COUNTS_SEG = 8;      // counts[8]: sorted entries per k_accumulate thread (counts[0] = valid entries, [1..7] = fold level sizes)

// counts[] of a sorted list of M valid entries (one device thread): the entries per accumulation thread, target T, fitted so
// that the grid is a whole number of waves of `wave` resident threads (MsmSorted comment; wave = 0: T as is), and the
// level sizes of the fold cascade: level 0 always emits ceil(M/seg) heads; a level >= 1 with <= MSM_SEG inputs is the
// last one (single thread, everything folded into the buckets) and emits none.
__device__ inline void msm_fill_counts(uint64_t* out, uint64_t M, uint32_t T, uint32_t seg_lo, uint64_t wave) {
    out[0] = M;
    uint64_t seg = T;
    if (wave) {
        const uint64_t k = (M + wave * T - 1) / (wave * T);              // waves at the target size
        if (k && k <= 3) seg = (M + k * wave - 1) / (k * wave);       // with 4+ waves the partial last wave still saturates the pipe (measured: no gain, more heads)
        if (seg < seg_lo) seg = seg_lo;
        if (seg > T) seg = T;
    }
    out[MSM_COUNTS_SEG] = seg;
    uint64_t m = (M + seg - 1) / seg;
    out[1] = m;
    for (int l = 2; l < 8; l++) { m = (m <= MSM_SEG) ? 0 : (m + MSM_SEG - 1) / MSM_SEG; out[l] = m; }
}


// Window-size choice.  Cost model: W_eff*n mixed adds (10 modmul) + one pass over the buckets (~60 modmul each);
// buckets = 2^(c-1) per window, shared by all windows in the precomputed-table mode.  `fr_bits` is the bit length of
// the scalar field (254 / 255): field-element scalars leave the windows above it empty, and the top *occupied* window
// only has top_bits = fr_bits + 1 - (W_eff-1)*c significant bits, i.e. it funnels all n terms into 2^top_bits buckets.
// Candidates whose top window is more than 32x denser than the others are skipped (giant buckets are handled
// correctly by the fold cascade, but cost latency-bound milliseconds).  W itself always covers 8*scalar_bytes + 1 bits,
// so arbitrary scalars (the reference accepts any value < 2^(8*sScalar)) stay correct.
__host__ inline MsmGeom msm_choose(uint64_t n, uint32_t scalar_bytes, int fr_bits, bool precomp) {
    int eff = (int)(8 * scalar_bytes) < fr_bits ? (int)(8 * scalar_bytes) : fr_bits;
    int best_c = 3; double best = 1e300;
    for (int c = 3; c <= 22; c++) {
        int weff = (eff + 1 + c - 1) / c, top = eff + 1 - (weff - 1) * c;
        if (weff > 1 && top < c - 5) continue;
        double buckets = (precomp ? 1.0 : (double)weff) * (double)(1u << (c - 1));
        double cost = (double)weff * (double)n * 10.0 + buckets * 60.0;
        if (cost < best) { best = cost; best_c = c; }
    }
    MsmGeom g; g.c = best_c; g.W = (int)((8 * scalar_bytes + 1 + best_c - 1) / best_c); g.B = 1u << (best_c - 1);
    return g;
}
// Precomputed-window mode (tables cover 32-byte scalars): all windows share one bucket set, so the bucket pass is
// cheap and what matters is the number of windows: take the largest c (fewest windows) that keeps the top window's
// density within 32x of the others and leaves on average >= ~W entries per bucket (2^(c-1) <= n).  Sparse buckets
// (a few dozen entries) also keep the per-thread head partials short-run, i.e. on the parallel k_fold_short path.
__host__ inline MsmGeom msm_geometry_precomp(uint64_t n_set, uint32_t scalar_bytes, int fr_bits = 254) {
    int l2 = 0; while ((1ull << (l2 + 1)) <= n_set) l2++;
    int cmax = l2; if (cmax > 22) cmax = 22; if (cmax < 8) cmax = 8;   // 2^(c-1) <= n/2: the bucket pass (1.3 ns/bucket) stays below ~1/3 of the accumulation (0.16 ns/entry)
    int c = 8;
    for (int cc = cmax; cc >= 8; cc--) {
        int weff = (fr_bits + 1 + cc - 1) / cc, top = fr_bits + 1 - (weff - 1) * cc;
        if (weff > 1 && top < cc - 5) continue;
        c = cc; break;
    }
    MsmGeom g; g.c = c; g.W = (int)((8 * scalar_bytes + 1 + c - 1) / c); g.B = 1u << (c - 1);
    g.precomp = 1; g.stride = n_set; g.first = 0;
    return g;
}
__host__ inline MsmGeom msm_geometry(uint64_t n, uint32_t scalar_bytes, int fr_bits = 254) {
    return msm_choose(n, scalar_bytes, fr_bits, false);
}

template <class F> __device__ __forceinline__ void load_affine(const Affine<F>* __restrict__ bases, uint32_t idx, F& x, F& y) {
    constexpr int NV = sizeof(F) / 16;
    const uint4* p = reinterpret_cast<const uint4*>(bases + idx);
    uint4* dx = reinterpret_cast<uint4*>(&x);
    uint4* dy = reinterpret_cast<uint4*>(&y);
#pragma unroll
    for (int k = 0; k < NV; k++) dx[k] = __ldg(p + k);
#pragma unroll
    for (int k = 0; k < NV; k++) dy[k] = __ldg(p + NV + k);
}
template <class T> __device__ __forceinline__ void store_vec(T* dst, const T& v) {
    constexpr int NV = sizeof(T) / 16;
    const uint4* s = reinterpret_cast<const uint4*>(&v);
    uint4* d = reinterpret_cast<uint4*>(dst);
#pragma unroll
    for (int k = 0; k < NV; k++) d[k] = s[k];
}
template <class T> __device__ __forceinline__ T load_vec(const T* src) {
    constexpr int NV = sizeof(T) / 16;
    T v; const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(&v);
#pragma unroll
    for (int k = 0; k < NV; k++) d[k] = s[k];
    return v;
}

// field inversion on the device: binary (Kaliski) for Fp, norm + binary for Fp2
template <class P> __device__ __forceinline__ Fp<P> PairInvF(const Fp<P>& a) { return Fp<P>::inv_binary(a); }
template <class P> __device__ __forceinline__ Fp2<P> PairInvF(const Fp2<P>& a) { return Fp2<P>::inv(a); }

// ------------------------------------------------------------------------------------------------
// level 0: affine bases gathered through the sorted (key, val) list
// ------------------------------------------------------------------------------------------------
template <class F, int MINB>
__global__ void __launch_bounds__(MSM_ACC_THREADS, MINB)
k_accumulate(const Affine<F>* __restrict__ bases, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
             const uint64_t* __restrict__ counts, XYZZ<F>* __restrict__ buckets,
             XYZZ<F>* __restrict__ heads, uint32_t* __restrict__ head_keys) {
    const uint64_t M = counts[0];
    const uint32_t seg = (uint32_t)counts[MSM_COUNTS_SEG];          // entries per thread, fitted to whole waves by k_count_valid
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint64_t lo = t * seg;
    if (lo >= M) return;
    uint64_t hi = lo + seg < M ? lo + seg : M;
    const F one = F::one();
    XYZZ<F> acc = XYZZ<F>::inf();
    uint32_t cur = keys[lo];
    bool first = true;
    for (uint64_t e = lo; e < hi; e++) {
        uint32_t k = keys[e], v = vals ? vals[e] : (uint32_t)e;
        if (k != cur) {
            if (first) { store_vec(heads + t, acc); head_keys[t] = cur; first = false; }
            else store_vec(buckets + cur, acc);
            acc = XYZZ<F>::inf(); cur = k;
        }
        F px, py;
        load_affine<F>(bases, v & 0x7fffffffu, px, py);
        if (!(px.is_zero() & py.is_zero())) {          // base at infinity contributes nothing (reference 6068-6086)
            py = F::cneg(py, (v >> 31) != 0);
            acc.add_affine(px, py, one);
        }
    }
    if (first) { store_vec(heads + t, acc); head_keys[t] = cur; }
    else store_vec(buckets + cur, acc);
}

// The same walk for an extension-field group with every point spread over a lane pair (Fp2L, ec.cuh): thread 2t holds the c0
// components of segment t's accumulator, thread 2t+1 the c1 components.  Half the registers per thread (the plain kernel needs
// 252 and runs 8 warps per SM), twice the threads; the arithmetic per point is the same 16 dual products + 4 multiplies, split
// evenly over the two lanes.  Memory layout is unchanged (x.c0 x.c1 y.c0 y.c1 zz.c0 ...): lane `par` moves the blocks 2k + par.
template <class T> struct fp2_param;
template <class P> struct fp2_param<Fp2<P>> { typedef P type; };
template <class P, int MINB>
__global__ void __launch_bounds__(MSM_ACC_THREADS, MINB)
k_accumulate_pair(const Affine<Fp2<P>>* __restrict__ bases, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                  const uint64_t* __restrict__ counts, XYZZ<Fp2<P>>* __restrict__ buckets,
                  XYZZ<Fp2<P>>* __restrict__ heads, uint32_t* __restrict__ head_keys) {
    typedef Fp2L<P> F; typedef Fp<P> B;
    const uint64_t M = counts[0];
    const uint32_t seg = (uint32_t)counts[MSM_COUNTS_SEG];
    const uint64_t t = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 1;
    const uint32_t par = threadIdx.x & 1u;
    uint64_t lo = t * seg;
    if (lo >= M) return;                                     // both lanes of a pair leave together
    uint64_t hi = lo + seg < M ? lo + seg : M;
    const F one = F::one();
    XYZZ<F> acc = XYZZ<F>::inf();
    auto put = [&](XYZZ<Fp2<P>>* dst, const XYZZ<F>& a) {
        B* q = reinterpret_cast<B*>(dst);
        store_vec(q + par, a.x.m); store_vec(q + 2 + par, a.y.m); store_vec(q + 4 + par, a.zz.m); store_vec(q + 6 + par, a.zzz.m);
    };
    uint32_t cur = keys[lo];
    bool first = true;
    for (uint64_t e = lo; e < hi; e++) {
        uint32_t k = keys[e], v = vals ? vals[e] : (uint32_t)e;
        if (k != cur) {
            if (first) { put(heads + t, acc); if (!par) head_keys[t] = cur; first = false; }
            else put(buckets + cur, acc);
            acc = XYZZ<F>::inf(); cur = k;
        }
        F px, py;
        {
            constexpr int NV = sizeof(B) / 16;
            const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const B*>(bases + (v & 0x7fffffffu)) + par);
            uint4* dx = reinterpret_cast<uint4*>(&px.m); uint4* dy = reinterpret_cast<uint4*>(&py.m);
#pragma unroll
            for (int i = 0; i < NV; i++) dx[i] = __ldg(p + i);
#pragma unroll
            for (int i = 0; i < NV; i++) dy[i] = __ldg(p + 2 * NV + i);
        }
        if (!(px.is_zero() & py.is_zero())) {
            py = F::cneg(py, (v >> 31) != 0);
            acc.add_affine(px, py, one);
        }
    }
    if (first) { put(heads + t, acc); if (!par) head_keys[t] = cur; }
    else put(buckets + cur, acc);
}

// ------------------------------------------------------------------------------------------------
// level 1 fast path: one thread per head partial.  Heads are sorted by key; a run of equal keys of length
// <= MSM_SHORT_RUN is summed by its first thread and added to the bucket (for uniform scalars practically every
// run has length 1, so this is one fully parallel read-modify-write per head).  Heads consumed here are marked
// INVALID in keys_out; longer runs (skewed scalars: giant buckets) keep their key and go to the k_fold cascade.
// ------------------------------------------------------------------------------------------------
static constexpr int MSM_SHORT_RUN = 8;
template <class F>
__global__ void __launch_bounds__(MSM_ACC_THREADS)
k_fold_short(const XYZZ<F>* __restrict__ heads, const uint32_t* __restrict__ keys_in, uint32_t* __restrict__ keys_out,
             const uint64_t* __restrict__ counts, XYZZ<F>* __restrict__ buckets) {
    const uint64_t M = counts[1];
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= M) return;
    const uint32_t k = keys_in[t];
    // locate the start of my run (looking back at most MSM_SHORT_RUN entries)
    uint64_t start = t; int back = 0;
    while (start > 0 && back < MSM_SHORT_RUN && keys_in[start - 1] == k) { start--; back++; }
    bool is_short = back < MSM_SHORT_RUN;
    uint64_t len = 0;
    if (is_short) {
        len = 1;
        while (start + len < M && len <= (uint64_t)MSM_SHORT_RUN && keys_in[start + len] == k) len++;
        is_short = len <= (uint64_t)MSM_SHORT_RUN;
    }
    keys_out[t] = is_short ? MSM_INVALID_KEY : k;
    if (!is_short || start != t) return;
    XYZZ<F> acc = load_vec(buckets + k);
    for (uint64_t e = 0; e < len; e++) { XYZZ<F> p = load_vec(heads + t + e); acc.add(p); }
    store_vec(buckets + k, acc);
}

// ------------------------------------------------------------------------------------------------
// level >= 1 cascade: fold the remaining head partials (sorted by key, INVALID = already consumed).
// `last` = single-thread final level.
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(MSM_ACC_THREADS)
k_fold(const XYZZ<F>* __restrict__ in, const uint32_t* __restrict__ in_keys, const uint64_t* __restrict__ counts, int level,
       XYZZ<F>* __restrict__ buckets, XYZZ<F>* __restrict__ heads, uint32_t* __restrict__ head_keys) {
    const uint64_t M = counts[level];
    const bool last = M <= MSM_SEG;
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint64_t lo = t * MSM_SEG;
    if (lo >= M) return;
    uint64_t hi = lo + MSM_SEG < M ? lo + MSM_SEG : M;
    XYZZ<F> acc = XYZZ<F>::inf();
    uint32_t cur = in_keys[lo];
    bool first = !last;
    auto flush = [&]() {
        if (first) { store_vec(heads + t, acc); head_keys[t] = cur; first = false; }
        else if (cur != MSM_INVALID_KEY) { XYZZ<F> b = load_vec(buckets + cur); b.add(acc); store_vec(buckets + cur, b); }
    };
    for (uint64_t e = lo; e < hi; e++) {
        uint32_t k = in_keys[e];
        if (k != cur) { flush(); acc = XYZZ<F>::inf(); cur = k; }
        if (k != MSM_INVALID_KEY) { XYZZ<F> p = load_vec(in + e); acc.add(p); }
    }
    flush();
}

// ------------------------------------------------------------------------------------------------
// bucket reduction.  Thread (w, j) owns buckets [j*L, (j+1)*L) of window w:
//   run = sum bucket[b],  sum = sum (b - j*L + 1) * bucket[b]   (running sums, reference _reduceTable
//   computes the same weighted sum by recursive halving), partial = sum + (j*L) * run.
// Then a shared-memory tree adds the partials of one CTA; CTAs of a window write to partials[w][cta].
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(128)
k_reduce(const XYZZ<F>* __restrict__ buckets, MsmGeom g, XYZZ<F>* __restrict__ partials, uint32_t ctas_per_window) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(smem_raw);
    const uint32_t w = blockIdx.x / ctas_per_window, cta = blockIdx.x % ctas_per_window;
    const uint32_t L = g.B < (uint32_t)MSM_RED_CHUNK ? g.B : MSM_RED_CHUNK;
    const uint32_t chunks = g.B / L;
    const uint32_t j = cta * blockDim.x + threadIdx.x;
    XYZZ<F> part = XYZZ<F>::inf();
    if (j < chunks) {
        const XYZZ<F>* bk = buckets + (uint64_t)w * g.B + (uint64_t)j * L;
        XYZZ<F> run = XYZZ<F>::inf(), sum = XYZZ<F>::inf();
        for (int b = (int)L - 1; b >= 0; b--) {
            XYZZ<F> p = load_vec(bk + b);
            run.add(p);
            sum.add(run);
        }
        // part = sum + (j*L) * run   (double-and-add, MSB first)
        uint32_t k = j * L;
        if (k) {
            int top = 31 - __clz(k);
            part = run;
            for (int bit = top - 1; bit >= 0; bit--) {
                part = XYZZ<F>::dbl(part);
                if ((k >> bit) & 1) part.add(run);
            }
        }
        part.add(sum);
    }
    store_vec(sm + threadIdx.x, part);
    __syncthreads();
    for (uint32_t s = blockDim.x >> 1; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            XYZZ<F> a = load_vec(sm + threadIdx.x), b = load_vec(sm + threadIdx.x + s);
            a.add(b);
            store_vec(sm + threadIdx.x, a);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) store_vec(partials + (uint64_t)w * ctas_per_window + cta, load_vec(sm));
}

// ------------------------------------------------------------------------------------------------
// Hierarchical bucket reduction (used when a window has >= 2048 buckets).  For a block of buckets [b0, b0+n):
//   R = sum B_b,   S = sum (b - b0 + 1) * B_b.
// m adjacent blocks of n buckets combine as  R = sum R_i,  S = sum S_i + n * sum_i i*R_i, where sum_i i*R_i is again a
// running sum (t += R_i; acc += t from the top).  So every level costs ~3 additions per child and log2(n) doublings
// per parent — no per-thread scalar multiply as in k_reduce (which spends ~40 % of its work there).
// k_reduce2: one CTA = 128 threads x 16 buckets (level 1) -> 16 groups of 8 -> 4 groups of 4 -> 1: (R, S) of 2048 buckets.
// k_window_sum2: one CTA per window folds the per-CTA (R, S) pairs, 8 at a time, down to the window total S.
// ------------------------------------------------------------------------------------------------
template <class F>
__device__ __forceinline__ void combine_children(const XYZZ<F>* Rin, const XYZZ<F>* Sin, int m, int log_n, XYZZ<F>& Rout, XYZZ<F>& Sout) {
    XYZZ<F> t = XYZZ<F>::inf(), acc = XYZZ<F>::inf(), ssum = load_vec(Sin);
    for (int i = m - 1; i >= 1; i--) {
        XYZZ<F> r = load_vec(Rin + i), s = load_vec(Sin + i);
        t.add(r); acc.add(t); ssum.add(s);
    }
    for (int k = 0; k < log_n; k++) acc = XYZZ<F>::dbl(acc);
    ssum.add(acc);
    XYZZ<F> r0 = load_vec(Rin); t.add(r0);
    Rout = t; Sout = ssum;
}

static constexpr int RED2_L = 16, RED2_THREADS = 128, RED2_BUCKETS = RED2_L * RED2_THREADS;   // 2048 buckets per CTA

template <class F>
__global__ void __launch_bounds__(RED2_THREADS)
k_reduce2(const XYZZ<F>* __restrict__ buckets, MsmGeom g, XYZZ<F>* __restrict__ outR, XYZZ<F>* __restrict__ outS) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(smem_raw);
    XYZZ<F>* R1 = sm; XYZZ<F>* S1 = sm + 128; XYZZ<F>* R2 = sm + 256; XYZZ<F>* S2 = sm + 272; XYZZ<F>* R3 = sm + 288; XYZZ<F>* S3 = sm + 292;
    const uint32_t tid = threadIdx.x;
    const XYZZ<F>* bk = buckets + (uint64_t)blockIdx.x * RED2_BUCKETS + (uint64_t)tid * RED2_L;
    {   // level 1: classic running sum over 16 buckets
        XYZZ<F> run = XYZZ<F>::inf(), sum = XYZZ<F>::inf();
        for (int b = RED2_L - 1; b >= 0; b--) { XYZZ<F> p = load_vec(bk + b); run.add(p); sum.add(run); }
        store_vec(R1 + tid, run); store_vec(S1 + tid, sum);
    }
    __syncthreads();
    if (tid < 16) { XYZZ<F> r, s; combine_children<F>(R1 + 8 * tid, S1 + 8 * tid, 8, 4, r, s); store_vec(R2 + tid, r); store_vec(S2 + tid, s); }   // n = 16
    __syncthreads();
    if (tid < 4) { XYZZ<F> r, s; combine_children<F>(R2 + 4 * tid, S2 + 4 * tid, 4, 7, r, s); store_vec(R3 + tid, r); store_vec(S3 + tid, s); }      // n = 128
    __syncthreads();
    if (tid == 0) { XYZZ<F> r, s; combine_children<F>(R3, S3, 4, 9, r, s); store_vec(outR + blockIdx.x, r); store_vec(outS + blockIdx.x, s); }      // n = 512
}

// per window: NC = B / 2048 pairs (power of two, <= 1024) -> S of the window.  One CTA of 128 threads per window.
template <class F>
__global__ void __launch_bounds__(128)
k_window_sum2(const XYZZ<F>* __restrict__ inR, const XYZZ<F>* __restrict__ inS, uint32_t NC, XYZZ<F>* __restrict__ out) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(smem_raw);     // two ping-pong regions of (R[128], S[128])
    const uint32_t tid = threadIdx.x;
    const XYZZ<F>* Rin = inR + (uint64_t)blockIdx.x * NC; const XYZZ<F>* Sin = inS + (uint64_t)blockIdx.x * NC;
    uint32_t n = NC; int log_block = 11;                    // a child covers 2^11 buckets at the first level
    int ping = 0;
    while (n > 1) {
        const uint32_t m = n >= 8 ? 8 : n, parents = n / m;
        XYZZ<F>* Rout = sm + ping * 256; XYZZ<F>* Sout = Rout + 128;
        for (uint32_t p = tid; p < parents; p += blockDim.x) {
            XYZZ<F> r, s; combine_children<F>(Rin + (uint64_t)p * m, Sin + (uint64_t)p * m, (int)m, log_block, r, s);
            store_vec(Rout + p, r); store_vec(Sout + p, s);
        }
        __syncthreads();
        Rin = Rout; Sin = Sout; n = parents; ping ^= 1;
        log_block += (m == 8 ? 3 : m == 4 ? 2 : 1);
    }
    if (tid == 0) store_vec(out + blockIdx.x, load_vec(Sin));
}

// one warp per window: lanes stride over the per-CTA partials of k_reduce, then a shared-memory tree
template <class F>
__global__ void __launch_bounds__(32)
k_window_sum(const XYZZ<F>* __restrict__ partials, uint32_t per_window, XYZZ<F>* __restrict__ out) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F>* sm = reinterpret_cast<XYZZ<F>*>(smem_raw);
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t i = threadIdx.x; i < per_window; i += 32) { XYZZ<F> p = load_vec(partials + (uint64_t)blockIdx.x * per_window + i); acc.add(p); }
    store_vec(sm + threadIdx.x, acc);
    __syncwarp();
    for (uint32_t s = 16; s > 0; s >>= 1) {
        if (threadIdx.x < s) { XYZZ<F> a = load_vec(sm + threadIdx.x), b = load_vec(sm + threadIdx.x + s); a.add(b); store_vec(sm + threadIdx.x, a); }
        __syncwarp();
    }
    if (threadIdx.x == 0) store_vec(out + blockIdx.x, load_vec(sm));
}

// ------------------------------------------------------------------------------------------------
// Bucket reduction, second design (default): axis sums + warp-shuffle weighted sums.
//
// The window sum  sum_b (b+1) * bucket[b]  is  T + sum_b b * bucket[b]  with T = sum of all buckets.  Write the bucket
// index as b = hi * 2^m + lo (a matrix of H rows by 2^m columns); with the row sums R_hi and the column sums C_lo
//     sum_b b * bucket[b] = 2^m * sum_hi hi * R_hi + sum_lo lo * C_lo,        T = sum_lo C_lo.
// Every bucket is added once into a row sum and once into a column sum (2 additions per bucket, the same count as the
// running-sum recursion of the reference's _reduceTable 5819-5907 or of k_reduce above), but the additions form plain
// trees: no per-thread scalar multiply and 4x the threads of k_reduce at the first level.
//   k_axis_sum   out[o][i] = sum_{s<S} in[o][s][i]  (S <= 8 per level; rows and columns of one level in one launch:
//                the row job views its rows as [S][len/S] so that both jobs read coalesced 128 B .. 4 KiB runs)
//   k_ws_chunks  one warp per 32 entries of R / C: lane l holds v_l; a shuffle suffix scan gives the suffix sums, their
//                shuffle-tree sum is sum_l l*v_l (weighted) and the first suffix sum is the plain total
//   k_ws_final   one CTA per window: the same warp routine over the chunk totals, then the power-of-two weights
//                (2^m, 2^5) by doublings of single points.
// ------------------------------------------------------------------------------------------------
template <class F> __device__ __noinline__ void padd(XYZZ<F>& a, const XYZZ<F>& b) { a.add(b); }

struct AxisJob { const void* in; void* out; uint64_t total; uint32_t S; uint32_t log_inner; };

template <class F>
__global__ void __launch_bounds__(128)
k_axis_sum(AxisJob j0, AxisJob j1) {
    const AxisJob j = blockIdx.y ? j1 : j0;
    const uint64_t gid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (gid >= j.total) return;
    const uint64_t o = gid >> j.log_inner, i = gid & ((1ull << j.log_inner) - 1);
    const XYZZ<F>* p = (const XYZZ<F>*)j.in + ((o * j.S) << j.log_inner) + i;
    XYZZ<F> acc = load_vec(p);
#pragma unroll 1
    for (uint32_t s = 1; s < j.S; s++) { XYZZ<F> v = load_vec(p + ((uint64_t)s << j.log_inner)); acc.add(v); }
    store_vec((XYZZ<F>*)j.out + gid, acc);
}

template <class F> __device__ __forceinline__ XYZZ<F> shfl_down_pt(const XYZZ<F>& v, int d) {
    constexpr int NW32 = sizeof(XYZZ<F>) / 4;
    union U { XYZZ<F> p; uint32_t w[NW32]; __device__ U() {} };
    U a, r; a.p = v;
#pragma unroll
    for (int k = 0; k < NW32; k++) r.w[k] = __shfl_down_sync(0xffffffffu, a.w[k], d);
    return r.p;
}
// lane l holds v_l.  Lane 0 receives T = sum_l v_l and W = sum_l l * v_l (all 32 lanes must call).
template <class F> __device__ __forceinline__ void warp_weighted_sum(XYZZ<F> v, XYZZ<F>& T, XYZZ<F>& W) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) { XYZZ<F> o = shfl_down_pt<F>(v, d); if (lane + d < 32) v.add(o); }   // suffix sums
    T = v;
    XYZZ<F> x = lane ? v : XYZZ<F>::inf();
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) { XYZZ<F> o = shfl_down_pt<F>(x, d); if (lane < d) x.add(o); }
    W = x;
}
template <class F> __device__ __forceinline__ XYZZ<F> warp_sum(XYZZ<F> x) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) { XYZZ<F> o = shfl_down_pt<F>(x, d); if (lane < d) x.add(o); }
    return x;
}

// vecR: [NW][lenR] (may be null / lenR = 0), vecC: [NW][lenC].  tw: [NW][nR + nC][2] = (T, W) of every 32-entry chunk.
template <class F>
__global__ void __launch_bounds__(128)
k_ws_chunks(const XYZZ<F>* __restrict__ vecR, uint32_t lenR, const XYZZ<F>* __restrict__ vecC, uint32_t lenC, uint32_t NW, XYZZ<F>* __restrict__ tw) {
    const uint32_t nR = (lenR + 31) / 32, nC = (lenC + 31) / 32, per = nR + nC;
    const uint32_t wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (wid >= NW * per) return;
    const uint32_t w = wid / per, jj = wid % per;
    const bool isR = jj < nR;
    const uint32_t j = isR ? jj : jj - nR, len = isR ? lenR : lenC, idx = j * 32 + lane;
    const XYZZ<F>* vec = (isR ? vecR : vecC) + (uint64_t)w * len;
    XYZZ<F> v = XYZZ<F>::inf();
    if (idx < len) v = load_vec(vec + idx);
    XYZZ<F> T, W;
    warp_weighted_sum<F>(v, T, W);
    if (lane == 0) { store_vec(tw + 2 * (uint64_t)wid, T); store_vec(tw + 2 * (uint64_t)wid + 1, W); }
}

// window sum = 2^(m+5) * a0 + 2^m * a1 + 2^5 * a2 + a3 + a4 with (chunk index j)
//   a0 = sum_j j * T^R_j,  a1 = sum_j W^R_j,  a2 = sum_j j * T^C_j,  a3 = sum_j W^C_j,  a4 = sum_j T^C_j (= all buckets).
// One CTA of four warps per window writes the five parts out[5 w + k]; the power-of-two weights (m + 10 doublings of single
// points: pure latency here) are applied by the host (msm_group.inl combine).
template <class F>
__global__ void __launch_bounds__(128)
k_ws_final(const XYZZ<F>* __restrict__ tw, uint32_t nR, uint32_t nC, XYZZ<F>* __restrict__ out) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, per = nR + nC;
    const XYZZ<F>* base = tw + 2 * (uint64_t)blockIdx.x * per;
    const bool r_side = warp < 2;
    const uint32_t cnt = r_side ? nR : nC, off = r_side ? 0 : nR;
    XYZZ<F> v = XYZZ<F>::inf();
    if (lane < cnt) v = load_vec(base + 2 * (uint64_t)(off + lane) + (warp & 1));   // even warps: T entries, odd warps: W entries
    XYZZ<F>* o = out + 5 * (uint64_t)blockIdx.x;
    if ((warp & 1) == 0) {
        XYZZ<F> tot, res;
        warp_weighted_sum<F>(v, tot, res);
        if (lane == 0) { store_vec(o + (r_side ? 0 : 2), res); if (!r_side) store_vec(o + 4, tot); }
    } else {
        XYZZ<F> res = warp_sum<F>(v);
        if (lane == 0) store_vec(o + (r_side ? 1 : 3), res);
    }
}

// One warp per output: out[o][i] = sum_{s<S} in[o][s][i], S <= 128: lane l adds s = l, l + 32, ... and a shuffle tree joins
// the lanes.  Used for everything the first axis-sum level leaves (2^16 partials per chain at 2^19 buckets): the work is
// negligible there and the latency (<= 3 + 5 dependent additions) is what counts.
template <class F>
__global__ void __launch_bounds__(128)
k_axis_tree(AxisJob j0, AxisJob j1) {
    const AxisJob j = blockIdx.y ? j1 : j0;
    const uint64_t wid = blockIdx.x * (uint64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    if (wid >= j.total) return;
    const uint64_t o = wid >> j.log_inner, i = wid & ((1ull << j.log_inner) - 1);
    const XYZZ<F>* p = (const XYZZ<F>*)j.in + ((o * j.S) << j.log_inner) + i;
    XYZZ<F> acc = XYZZ<F>::inf();
#pragma unroll 1
    for (uint32_t s = lane; s < j.S; s += 32) { XYZZ<F> v = load_vec(p + ((uint64_t)s << j.log_inner)); acc.add(v); }
    acc = warp_sum<F>(acc);
    if (lane == 0) store_vec((XYZZ<F>*)j.out + wid, acc);
}

// Host plan of the axis-sum levels for one geometry.  Buckets of a window form H = 2^er rows... of 2^m columns
// (m = WS_COL_BITS when the window has more than 2^m buckets, else there is no split and C = the buckets themselves).
static constexpr int WS_COL_BITS = 10;
struct WsPlan {
    bool ok = false;                 // false: geometry outside the design (more than 2^20 buckets per window) -> k_reduce
    int m = 0, er = 0, ec = 0;       // column bits, bits the row chain reduces (= m), bits the column chain reduces
    int levels = 0; int br[8] = {0}, bc[8] = {0};
    uint32_t lenR = 0, lenC = 0, nR = 0, nC = 0;
    size_t rowA = 0, rowB = 0, colA = 0, colB = 0, tw = 0;   // scratch sizes in XYZZ elements
    size_t elems() const { return rowA + rowB + colA + colB + tw + 8; }
};
__host__ inline WsPlan ws_plan(const MsmGeom& g) {
    WsPlan p; const int cbits = g.c - 1; const size_t NW = g.windows();
    if (cbits > 2 * WS_COL_BITS || cbits < 0) return p;
    p.ok = true;
    if (cbits > WS_COL_BITS) { p.m = WS_COL_BITS; p.er = p.m; p.ec = cbits - p.m; p.lenR = 1u << p.ec; p.lenC = 1u << p.m; }
    else { p.lenR = 0; p.lenC = g.B; }
    // level 0: S = 8 (k_axis_sum, carries the work); level 1: everything left, <= 7 bits (k_axis_tree, one warp per output)
    int rr = p.er, rc = p.ec;
    for (int l = 0; l < 2 && (rr > 0 || rc > 0); l++) {
        p.levels++;
        p.br[l] = l == 0 ? (rr < 3 ? rr : 3) : rr; p.bc[l] = l == 0 ? (rc < 3 ? rc : 3) : rc; rr -= p.br[l]; rc -= p.bc[l];
        const size_t orow = p.br[l] ? (NW * g.B) >> (p.er - rr) : 0, ocol = p.bc[l] ? (NW * g.B) >> (p.ec - rc) : 0;
        if (l & 1) { p.rowB = orow; p.colB = ocol; } else { p.rowA = orow; p.colA = ocol; }
    }
    p.nR = (p.lenR + 31) / 32; p.nC = (p.lenC + 31) / 32;
    p.tw = 2 * NW * (p.nR + p.nC);
    return p;
}
// scratch (in XYZZ elements) of the reduction: k_reduce partials, or the axis-sum ping-pong buffers + chunk pairs
__host__ inline size_t msm_reduce_scratch_elems(const MsmGeom& g) {
    const uint32_t NW = g.windows();
    const uint32_t L = g.B < (uint32_t)MSM_RED_CHUNK ? g.B : MSM_RED_CHUNK;
    const uint32_t ctas_per_window = (g.B / L + 127) / 128;
    const size_t legacy = (size_t)2 * NW * ctas_per_window;
    const WsPlan p = ws_plan(g);
    return (p.ok && p.elems() > legacy) ? p.elems() : legacy;
}

// ------------------------------------------------------------------------------------------------
// Precomputed window multiples for a registered base set: table[w*n + i] = 2^(c*w) * P_i (affine), w < W.
// One thread per point: c doublings per window in XYZZ, one inversion per table entry.  One-time cost per key.
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(128) k_precompute(const Affine<F>* __restrict__ bases, uint64_t n, int c, int W, Affine<F>* __restrict__ table) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> a = load_vec(bases + i);
    store_vec(table + i, a);
    if (a.is_inf()) {
        for (int w = 1; w < W; w++) store_vec(table + (uint64_t)w * n + i, a);
        return;
    }
    XYZZ<F> p; p.x = a.x; p.y = a.y; p.zz = F::one(); p.zzz = F::one();
    for (int w = 1; w < W; w++) {
        for (int j = 0; j < c; j++) p = XYZZ<F>::dbl(p);
        Affine<F> o;
        if (p.is_inf()) { o.x = F::zero(); o.y = F::zero(); }
        else { F t = PairInvF(F::mul(p.zz, p.zzz)); o.x = F::mul(p.x, F::mul(t, p.zzz)); o.y = F::mul(p.y, F::mul(t, p.zz)); p.x = o.x; p.y = o.y; p.zz = F::one(); p.zzz = F::one(); }
        store_vec(table + (uint64_t)w * n + i, o);
    }
}

// ------------------------------------------------------------------------------------------------
// Synthetic bases for benchmarks and tests, written as affine Montgomery points.  The definition is the CPU
// oracle's incremental generator (chunks of 4096 points: P_{c,0} = k0(c)*G, P_{c,j+1} = P_{c,j} + kd*G), which costs the
// host two additions per point; here every point is computed independently as (k0(c) + j*kd)*G — the same group
// element, hence the same affine bytes — so the B200 arm and the CPU reference arm of bench.py build identical keys.
// One thread per point: 77-bit double-and-add in XYZZ, then one field inversion.
__host__ __device__ inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull; x = (x ^ (x >> 27)) * 0x94D049BB133111EBull; return x ^ (x >> 31);
}
static constexpr uint64_t GEN_CHUNK = 4096;
template <class F>
__global__ void __launch_bounds__(128) k_gen_points(Affine<F> g, uint64_t seed, uint64_t n, Affine<F>* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t c = i / GEN_CHUNK, j = i % GEN_CHUNK;
    const uint64_t k0 = (seed ^ 0x9E3779B97F4A7C15ull) + c * 0xD1B54A32D192ED03ull, kd = seed * 2654435761ull + 12345ull;
    // s = k0 + j*kd  (< 2^77) as (hi, lo)
    uint64_t lo = j * kd, hi = __umul64hi(j, kd);
    lo += k0; hi += lo < k0 ? 1 : 0;
    const F one = F::one();
    XYZZ<F> r = XYZZ<F>::inf();
    for (int bit = 79; bit >= 0; bit--) {
        r = XYZZ<F>::dbl(r);
        const uint64_t wd = bit >= 64 ? hi : lo;
        if ((wd >> (bit & 63)) & 1) r.add_affine(g.x, g.y, one);
    }
    Affine<F> a;
    if (r.is_inf()) { a.x = F::zero(); a.y = F::zero(); }
    else { F t = PairInvF(F::mul(r.zz, r.zzz)); a.x = F::mul(r.x, F::mul(t, r.zzz)); a.y = F::mul(r.y, F::mul(t, r.zz)); }
    store_vec(out + i, a);
}

}  // namespace sb
#include "msm_pair.cuh"
namespace sb {

// ------------------------------------------------------------------------------------------------
// Device scratch (grow-only) and the two halves of the pipeline.
// ------------------------------------------------------------------------------------------------
struct MsmScratch {
    void* p = nullptr; size_t cap = 0;
    void* get(size_t bytes) {
        if (bytes > cap) { if (p) cudaFree(p); p = nullptr; cap = 0; if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr; cap = bytes; }
        return p;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

extern int g_msm_tuning[12];

struct MsmLaunchStats {
    int launches = 0;
    // optional profiling: event pairs recorded around kernel groups (tag = PROF_* below; accumulation uses cur_tag)
    cudaEvent_t* ev = nullptr; int nev = 0; int used = 0; int tag[128] = {0}; int cur_tag = 0;
};
// PROF_PAIR_G1/G2: batched-affine rounds, counted as accumulation time of the group but not as an accumulation launch
enum { PROF_ACC_G1 = 1, PROF_ACC_G2 = 2, PROF_SORT = 3, PROF_FOLD = 4, PROF_REDUCE = 5, PROF_QAP = 6, PROF_NTT = 7, PROF_JOIN = 8,
       PROF_PAIR_G1 = 9, PROF_PAIR_G2 = 10 };
// one event pair around a group of launches on `st`; a no-op unless profiling is armed (api.cu prof_begin)
struct ProfScope {
    MsmLaunchStats* s; cudaStream_t st; int idx = -1;
    ProfScope(MsmLaunchStats* s_, int tag, cudaStream_t st_) : s(s_), st(st_) {
        if (s && s->ev && s->used + 2 <= s->nev && s->used / 2 < 128) { idx = s->used; s->used += 2; s->tag[idx / 2] = tag; cudaEventRecord(s->ev[idx], st); }
    }
    void end() { if (idx >= 0) { cudaEventRecord(s->ev[idx + 1], st); idx = -1; } }
    void end(cudaStream_t other) { st = other; end(); }
};

// Sorted digit entries of one scalar vector; shared by every MSM that uses the same scalars
// (Groth16: A, B1, B2 and C all multiply the witness, src/groth16_prove.js:84-97).
struct MsmSorted {
    const uint32_t* keys = nullptr; const uint32_t* vals = nullptr; const uint64_t* counts = nullptr;
    uint64_t n = 0, total = 0; MsmGeom g{};
    // Sorted entries per k_accumulate thread.  The target is MSM_SEG, or more when the buckets are dense (hundreds of entries
    // per bucket, e.g. the 9n-point fflonk commitments: a thread's first run becomes a head partial, and with several heads
    // per bucket the runs of equal head keys outgrow k_fold_short's parallel path).  The actual value is chosen on the
    // device (k_count_valid, counts[MSM_COUNTS_SEG]) once the number of valid entries M is known: every thread does the same
    // work, so the kernel time is waves x seg, and seg = ceil(M / (k * resident threads)) makes the grid exactly k full waves
    // of the 148 SMs instead of k - 1 waves and a fraction (applied for k <= 3: shards of a multi-GPU proof, small MSMs;
    // measured on the 2-GPU shards: G1 accumulation -7.5 %, G2 -10.6 %; with more waves the effect vanishes).  seg_lo = the smallest value the device may pick (grid and
    // head-buffer sizing on the host).
    uint32_t seg_lo = MSM_SEG;
};

// msm_sort.cu: SM count of the current device, output positions of a batched-affine round (non-template part)
int msm_sm_count();
size_t msm_pair_scan_tmp_bytes(uint64_t items);
int msm_pair_scan(const uint32_t* counts, uint32_t* pos, uint64_t items, void* tmp, size_t tmp_bytes, cudaStream_t stream);

// msm_sort.cu: digits + radix sort + valid count.  d_scalars is a device pointer.
int msm_sort_entries(const uint8_t* d_scalars, uint32_t sbytes, uint64_t n, MsmGeom g, MsmScratch& scratch,
                     cudaStream_t stream, MsmSorted* out, MsmLaunchStats* stats);

// Scratch layout of msm_buckets_impl (byte offsets from its scratch_off) for a list of at most `total` entries.
struct MsmBucketLayout { uint64_t heads0 = 0; size_t headsA = 0, hkA = 0, headsB = 0, hkB = 0, hkM = 0, part = 0, bytes = 0; };
template <class F>
MsmBucketLayout msm_bucket_layout(const MsmGeom& g, uint64_t total, uint32_t seg_lo) {
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    MsmBucketLayout L;
    L.heads0 = (total + seg_lo - 1) / seg_lo;   // upper bound; the device knows the exact count (counts[1])
    const uint64_t heads1 = (L.heads0 + MSM_SEG - 1) / MSM_SEG;
    L.headsA = al((uint64_t)g.windows() * g.B * sizeof(XYZZ<F>)); L.hkA = L.headsA + al(L.heads0 * sizeof(XYZZ<F>));
    L.headsB = L.hkA + al(L.heads0 * 4); L.hkB = L.headsB + al(heads1 * sizeof(XYZZ<F>));
    L.hkM = L.hkB + al(heads1 * 4);                       // level-1 keys after the short-run fast path
    L.part = L.hkM + al(L.heads0 * 4);
    L.bytes = L.part + al(msm_reduce_scratch_elems(g) * sizeof(XYZZ<F>));
    return L;
}

// Bucket accumulation + reduction for one base set.  Writes g.W window sums to d_wsum (device).  Asynchronous.
// If tail_stream differs from stream, the throughput-bound accumulation runs on `stream` and the latency-bound tail
// (fold, bucket reduction, window sum) on `tail_stream` after `ev_acc` (recorded here): with a higher-priority tail
// stream the tail of one MSM slips into the SM slots freed by the next MSM's accumulation instead of queueing behind it.
template <class F>
int msm_buckets_impl(const Affine<F>* d_bases, const MsmSorted& s, MsmScratch& scratch, size_t scratch_off, cudaStream_t stream,
                     XYZZ<F>* d_wsum, MsmLaunchStats* stats, cudaStream_t tail_stream, cudaEvent_t ev_acc);

// Entry: batched-affine rounds (msm_pair.cuh) shrink the sorted list first where they pay, then the segmented XYZZ
// pipeline runs on what is left.  The rounds are the default for BN254 G2 (an XYZZ mixed addition costs 27.5
// modmul-equivalents there) on lists of >= PAIR_MIN_ENTRIES entries that average more than PAIR_STOP_DENSITY entries per
// bucket (precomputed-table MSMs: 26 or more per bucket).  Measured on a B200
// (1000 W), one registered 2^20 BN254 MSM, uniform scalars (profiles/ab_batch_affine.py, profiles/README.md):
//   G2: XYZZ only 10.18 ms, 1 round 9.30, 2 rounds 8.96, 3 rounds 9.02, 4 rounds 9.23 -> stop at ~8 entries per bucket;
//   G1: XYZZ only 3.24 ms, 1 round 3.39, 2 rounds 3.49 -> the rounds stay off (9.5 modmul per XYZZ addition is too
//   close to the ~6 of an affine one plus the extra passes over memory).  BLS12-381 G2 has not been measured: off.
// sb_set_tuning(4, 2) forces the rounds (at least one, and down to PAIR_FORCED_STOP_DENSITY), (4, 1) turns them off,
// (5, R) caps their number.
static constexpr double PAIR_STOP_DENSITY = 8.0;     // rounds run while the list averages more entries per bucket than this
static constexpr double PAIR_FORCED_STOP_DENSITY = 2.0;
static constexpr uint64_t PAIR_MIN_ENTRIES = 1ull << 20;
static constexpr int PAIR_MAX_ROUNDS = 8;
static constexpr uint64_t PAIR_MAX_SLOTS = 64;       // pair slots per thread
template <class F> struct PairDefault { static constexpr bool value = false; };
template <> struct PairDefault<Fp2<BnFq>> { static constexpr bool value = true; };

template <class F>
int msm_buckets(const Affine<F>* d_bases, const MsmSorted& s, MsmScratch& scratch, cudaStream_t stream,
                XYZZ<F>* d_wsum, MsmLaunchStats* stats, cudaStream_t tail_stream = nullptr, cudaEvent_t ev_acc = nullptr) {
    const MsmGeom g = s.g;
    const uint64_t NB = (uint64_t)g.windows() * g.B;
    const int mode = g_msm_tuning[4];
    const double stop = mode == 2 ? PAIR_FORCED_STOP_DENSITY : PAIR_STOP_DENSITY;
    const bool dense = NB && (double)s.total > PAIR_STOP_DENSITY * (double)NB;
    const bool use = mode == 2 || (mode == 0 && PairDefault<F>::value && s.total >= PAIR_MIN_ENTRIES && dense);
    if (!use || s.total == 0 || NB >= (1ull << 31) || s.total >= (1ull << 31))
        return msm_buckets_impl<F>(d_bases, s, scratch, 0, stream, d_wsum, stats, tail_stream, ev_acc);
    // Round plan on host upper bounds (the device knows the exact lengths): a round turns n entries into at most
    // ceil(n/2) + (key changes) <= ceil(n/2) + min(NB, n); it is expected to leave n/2 + NB/2 (half the buckets end on an
    // odd position).  Every round gets ~2048 threads per SM (several waves of both round kernels) and 1..64 slots per thread.
    uint64_t ub[PAIR_MAX_ROUNDS + 1], Jub[PAIR_MAX_ROUNDS], T[PAIR_MAX_ROUNDS]; uint32_t K[PAIR_MAX_ROUNDS];
    const uint64_t target = (uint64_t)msm_sm_count() * 2048;
    double est = (double)s.total;
    int R = 0; ub[0] = s.total;
    while (R < PAIR_MAX_ROUNDS && (est > stop * (double)NB || (R == 0 && mode == 2))) {
        Jub[R] = (ub[R] + 1) / 2;
        uint64_t k = (Jub[R] + target) / target; if (k > PAIR_MAX_SLOTS) k = PAIR_MAX_SLOTS;
        K[R] = (uint32_t)k;
        T[R] = ((Jub[R] + k) / k + PAIR_THREADS - 1) / PAIR_THREADS * PAIR_THREADS;    // K * T >= Jub + 1 slots
        ub[R + 1] = std::min(ub[R], (ub[R] + 1) / 2 + std::min(NB, ub[R]));
        est = est / 2 + (double)NB / 2;
        R++;
    }
    if (g_msm_tuning[5] > 0 && g_msm_tuning[5] < R) R = g_msm_tuning[5];
    uint64_t Tmax = 0; for (int r = 0; r < R; r++) Tmax = std::max(Tmax, T[r]);
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t scan_tmp = msm_pair_scan_tmp_bytes(Jub[0] + 1);
    const size_t o_outc = al((size_t)R * 128), o_pos = o_outc + al((Jub[0] + 1) * 4), o_tmp = o_pos + al((Jub[0] + 1) * 4);
    const size_t o_pre = o_tmp + al(scan_tmp), o_tp = o_pre + al(Jub[0] * sizeof(F)), o_inv = o_tp + al(Tmax * sizeof(F));
    const size_t o_P0 = o_inv + al(Tmax * sizeof(F)), o_P1 = o_P0 + al(ub[1] * sizeof(Affine<F>)), o_K0 = o_P1 + al(ub[1] * sizeof(Affine<F>));
    const size_t o_K1 = o_K0 + al(ub[1] * 4), o_rest = o_K1 + al(ub[1] * 4);
    MsmSorted s2 = s; s2.total = ub[R]; s2.vals = nullptr; s2.seg_lo = MSM_SEG / 2;       // k_pair_invert's count fit
    // one allocation for the rounds and the pipeline behind them: the scratch must not be reallocated while the rounds use it
    if (!scratch.get(o_rest + msm_bucket_layout<F>(g, s2.total, s2.seg_lo).bytes)) return (int)cudaErrorMemoryAllocation;
    uint8_t* base = (uint8_t*)scratch.p;
    uint32_t* outc = (uint32_t*)(base + o_outc); uint32_t* pos = (uint32_t*)(base + o_pos);
    F* pre = (F*)(base + o_pre); F* tprod = (F*)(base + o_tp); F* invp = (F*)(base + o_inv);
    Affine<F>* P[2] = {(Affine<F>*)(base + o_P0), (Affine<F>*)(base + o_P1)};
    uint32_t* Kb[2] = {(uint32_t*)(base + o_K0), (uint32_t*)(base + o_K1)};
    const uint64_t wave = (uint64_t)msm_sm_count() * 4 * MSM_ACC_THREADS;
    int launches = 0;
    ProfScope prof(stats, stats && stats->cur_tag == PROF_ACC_G1 ? PROF_PAIR_G1 : PROF_PAIR_G2, stream);
    const Affine<F>* src = d_bases; const uint32_t* keys = s.keys; const uint64_t* cin = s.counts;
    for (int r = 0; r < R; r++) {
        uint64_t* cout = (uint64_t*)(base + (size_t)r * 128);
        const unsigned grid = (unsigned)(T[r] / PAIR_THREADS), igrid = (unsigned)((T[r] / PAIR_LANE_PRODUCTS + 127) / 128);
        if (r == 0) k_pair_prefix<F, true><<<grid, PAIR_THREADS, 0, stream>>>(src, s.vals, keys, cin, Jub[r], K[r], pre, tprod, outc);
        else k_pair_prefix<F, false><<<grid, PAIR_THREADS, 0, stream>>>(src, nullptr, keys, cin, Jub[r], K[r], pre, tprod, outc);
        int rc = msm_pair_scan(outc, pos, Jub[r] + 1, base + o_tmp, scan_tmp, stream);
        if (rc) return rc;
        k_pair_invert<F><<<igrid, 128, 0, stream>>>(tprod, T[r], invp, pos, Jub[r], cout, wave);
        if (r == 0) k_pair_apply<F, true><<<grid, PAIR_THREADS, 0, stream>>>(src, s.vals, keys, cin, K[r], pre, invp, pos, P[0], Kb[0]);
        else k_pair_apply<F, false><<<grid, PAIR_THREADS, 0, stream>>>(src, nullptr, keys, cin, K[r], pre, invp, pos, P[r & 1], Kb[r & 1]);
        launches += 5;   // prefix, scan (2), invert, apply
        src = P[r & 1]; keys = Kb[r & 1]; cin = cout;
    }
    prof.end();
    if (stats) stats->launches += launches;
    s2.keys = keys; s2.counts = cin;
    return msm_buckets_impl<F>(src, s2, scratch, o_rest, stream, d_wsum, stats, tail_stream, ev_acc);
}

template <class F>
int msm_buckets_impl(const Affine<F>* d_bases, const MsmSorted& s, MsmScratch& scratch, size_t scratch_off, cudaStream_t stream,
                     XYZZ<F>* d_wsum, MsmLaunchStats* stats, cudaStream_t tail_stream, cudaEvent_t ev_acc) {
    const MsmGeom g = s.g;
    const uint32_t NW = g.windows();
    const uint64_t nbuckets = (uint64_t)NW * g.B;
    const uint32_t L = g.B < (uint32_t)MSM_RED_CHUNK ? g.B : MSM_RED_CHUNK;
    const uint32_t chunks = g.B / L;
    const uint32_t red_threads = 128;
    const uint32_t ctas_per_window = (chunks + red_threads - 1) / red_threads;
    const MsmBucketLayout lay = msm_bucket_layout<F>(g, s.total, s.seg_lo);
    const uint64_t heads0 = lay.heads0;
    uint8_t* base = (uint8_t*)scratch.get(scratch_off + lay.bytes);
    if (!base) return (int)cudaErrorMemoryAllocation;
    base += scratch_off;
    XYZZ<F>* buckets = (XYZZ<F>*)base;
    XYZZ<F>* headsA = (XYZZ<F>*)(base + lay.headsA); uint32_t* hkA = (uint32_t*)(base + lay.hkA);
    XYZZ<F>* headsB = (XYZZ<F>*)(base + lay.headsB); uint32_t* hkB = (uint32_t*)(base + lay.hkB);
    XYZZ<F>* partials = (XYZZ<F>*)(base + lay.part);
    uint32_t* hkM = (uint32_t*)(base + lay.hkM);
    int launches = 0;
    cudaMemsetAsync(buckets, 0, nbuckets * sizeof(XYZZ<F>), stream);
    if (heads0) {
        ProfScope prof(stats, stats ? stats->cur_tag : 0, stream);
        {
            const unsigned grid = (unsigned)((heads0 + MSM_ACC_THREADS - 1) / MSM_ACC_THREADS);
            // occupancy variants (sb_set_tuning(0, minBlocksPerSM)): base-field groups run best at 4 CTAs/SM (124 regs);
            // extension-field groups (accumulator = 64-96 registers) have their own variants
            constexpr bool ext = sizeof(F) > 48 && (sizeof(F) % 64 == 0 || sizeof(F) == 96);
            if constexpr (ext) {
                typedef typename fp2_param<F>::type FP;
                const unsigned pgrid = (unsigned)((2 * heads0 + MSM_ACC_THREADS - 1) / MSM_ACC_THREADS);
                if (g_msm_tuning[9] == 4) k_accumulate_pair<FP, 4><<<pgrid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA);
                else if (g_msm_tuning[9] == 3) k_accumulate_pair<FP, 3><<<pgrid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA);
                else switch (g_msm_tuning[0]) {
                case 3: k_accumulate<F, 3><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                case 4: k_accumulate<F, 4><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                default: k_accumulate<F, 2><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;   // measured best: 8.0 ms vs 8.5 (2^20 G2)
                }
            } else if constexpr (sizeof(F) > 32) {
                // 12-limb base field (BLS12-381 G1).  At 4 CTAs/SM the 128-register cap spills ~50 words of the mixed addition
                // (ptxas: 218 B spill stores / 188 B loads); 3 CTAs/SM (168 registers) and 2 (190) do not spill.  Measured on the
                // B200 (PLONK 2^18, nine accumulations): 2 CTAs/SM 15.8 ms, 4 CTAs/SM 16.7 ms, 3 CTAs/SM 19.3 ms
                // (profiles/ab_r2_summary.txt) -> 2 is the default; sb_set_tuning(10, 3 | 4) selects the others.
                switch (g_msm_tuning[8]) {
                case 4: k_accumulate<F, 4><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                case 3: k_accumulate<F, 3><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                default: k_accumulate<F, 2><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                }
            } else {
                // 8-limb base field (BN254 G1): 122 registers at 4 CTAs/SM, no spills; sb_set_tuning(12, 3 | 2) = lower-occupancy builds
                switch (g_msm_tuning[10]) {
                case 3: k_accumulate<F, 3><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                case 2: k_accumulate<F, 2><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                default: k_accumulate<F, 4><<<grid, MSM_ACC_THREADS, 0, stream>>>(d_bases, s.keys, s.vals, s.counts, buckets, headsA, hkA); break;
                }
            }
            launches++;
        }
        prof.end();
        if (tail_stream && tail_stream != stream && ev_acc) {
            cudaEventRecord(ev_acc, stream); cudaStreamWaitEvent(tail_stream, ev_acc, 0); stream = tail_stream;
        }
        ProfScope pfold(stats, PROF_FOLD, stream);
        k_fold_short<F><<<(unsigned)((heads0 + MSM_ACC_THREADS - 1) / MSM_ACC_THREADS), MSM_ACC_THREADS, 0, stream>>>(
            headsA, hkA, hkM, s.counts, buckets); launches++;
        // fold cascade: level l consumes counts[l] heads (upper bound m on the host, exact count on the device)
        uint64_t m = heads0; int level = 1;
        XYZZ<F>* hin = headsA; uint32_t* kin = hkM; XYZZ<F>* hout = headsB; uint32_t* kout = hkB;
        while (true) {
            uint64_t threads = (m + MSM_SEG - 1) / MSM_SEG;
            k_fold<F><<<(unsigned)((threads + MSM_ACC_THREADS - 1) / MSM_ACC_THREADS), MSM_ACC_THREADS, 0, stream>>>(
                hin, kin, s.counts, level, buckets, hout, kout); launches++;
            if (m <= (uint64_t)MSM_SEG) break;
            m = threads; level++;
            XYZZ<F>* th = hin; hin = hout; hout = th; uint32_t* tk = kin; kin = kout; kout = tk;
            if (level >= 8) return (int)cudaErrorUnknown;
        }
        pfold.end();
    }
    if (!heads0 && tail_stream && tail_stream != stream && ev_acc) { cudaEventRecord(ev_acc, stream); cudaStreamWaitEvent(tail_stream, ev_acc, 0); stream = tail_stream; }
    ProfScope pred(stats, PROF_REDUCE, stream);
    const WsPlan wp = ws_plan(g);
    if (wp.ok && g_msm_tuning[1] == 0) {
        // axis sums (rows and columns of one level per launch), then the warp-shuffle weighted sums
        XYZZ<F>* rowb[2] = {partials, partials + wp.rowA};
        XYZZ<F>* colb[2] = {partials + wp.rowA + wp.rowB, partials + wp.rowA + wp.rowB + wp.colA};
        XYZZ<F>* tw = partials + wp.rowA + wp.rowB + wp.colA + wp.colB;
        const XYZZ<F>* rin = buckets; const XYZZ<F>* cin = buckets;
        int rr = wp.er, rc = wp.ec;
        for (int l = 0; l < wp.levels; l++) {
            AxisJob jr{nullptr, nullptr, 0, 1, 0}, jc{nullptr, nullptr, 0, 1, 0};
            if (wp.br[l]) { rr -= wp.br[l]; jr = AxisJob{rin, rowb[l & 1], (uint64_t)nbuckets >> (wp.er - rr), 1u << wp.br[l], (uint32_t)rr}; rin = rowb[l & 1]; }
            if (wp.bc[l]) { rc -= wp.bc[l]; jc = AxisJob{cin, colb[l & 1], (uint64_t)nbuckets >> (wp.ec - rc), 1u << wp.bc[l], (uint32_t)wp.m}; cin = colb[l & 1]; }
            const uint64_t mx = jr.total > jc.total ? jr.total : jc.total;
            if (l == 0) k_axis_sum<F><<<dim3((unsigned)((mx + 127) / 128), 2), 128, 0, stream>>>(jr, jc);
            else k_axis_tree<F><<<dim3((unsigned)((mx + 3) / 4), 2), 128, 0, stream>>>(jr, jc);
            launches++;
        }
        const uint32_t per = wp.nR + wp.nC;
        k_ws_chunks<F><<<(NW * per + 3) / 4, 128, 0, stream>>>(wp.lenR ? rin : nullptr, wp.lenR, cin, wp.lenC, NW, tw); launches++;
        k_ws_final<F><<<NW, 128, 0, stream>>>(tw, wp.nR, wp.nC, d_wsum); launches++;
    } else if (g.B >= (uint32_t)RED2_BUCKETS && g.B / RED2_BUCKETS <= 1024 && g_msm_tuning[1] == 2) {   // experimental: less work (-36 %) but 2-3x the
        // dependent-add latency of k_reduce; measured slower (proof 27.4 ms vs 26.0 ms overlapped, 31.3 vs 26.6 serialised)
        // hierarchical reduction: per-CTA (R, S) pairs live in the partials area (2 * NC entries per window <= ctas_per_window)
        const uint32_t NC = g.B / RED2_BUCKETS;
        XYZZ<F>* pR = partials; XYZZ<F>* pS = partials + (size_t)NW * NC;
        static bool configured = false;
        if (!configured) {
            cudaFuncSetAttribute(k_reduce2<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(296 * sizeof(XYZZ<F>)));
            cudaFuncSetAttribute(k_window_sum2<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(512 * sizeof(XYZZ<F>)));
            configured = true;
        }
        k_reduce2<F><<<NW * NC, RED2_THREADS, 296 * sizeof(XYZZ<F>), stream>>>(buckets, g, pR, pS); launches++;
        k_window_sum2<F><<<NW, 128, 512 * sizeof(XYZZ<F>), stream>>>(pR, pS, NC, d_wsum); launches++;
    } else {
        k_reduce<F><<<NW * ctas_per_window, red_threads, red_threads * sizeof(XYZZ<F>), stream>>>(buckets, g, partials, ctas_per_window); launches++;
        k_window_sum<F><<<NW, 32, 32 * sizeof(XYZZ<F>), stream>>>(partials, ctas_per_window, d_wsum); launches++;
    }
    pred.end();
    if (stats) stats->launches += launches;
    return (int)cudaGetLastError();
}

}  // namespace sb
