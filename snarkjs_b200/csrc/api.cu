// api.cu — the C ABI of libsnarkb200.so (include/snarkb200.h): context, device buffers, table caches, the
// drop-in bulk operations, and the fused Groth16 prover.  Host-side orchestration only; kernels live in
// msm*.cu / fr_kernels.cu.  There is no CPU fallback: without a CUDA device sb_create fails.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <map>
#include <algorithm>
#include <mutex>
#include <future>
#include <thread>
#include <dlfcn.h>
#include <nccl.h>      // types and prototypes only: the library is dlopen'ed on first use (no link-time dependency)
#include <fcntl.h>
#include <unistd.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include "../../include/snarkb200.h"
#include "ec.cuh"
#include "msm.cuh"
#include "msm_entry.h"
#include "fr_entry.h"

using namespace sb;
namespace sb { double calibrate(int what, cudaStream_t stream); extern int g_ntt_tile_log; }

namespace {

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    void* get(size_t bytes) {
        if (bytes > cap) { if (p) cudaFree(p); p = nullptr; cap = 0; if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr; cap = bytes; }
        return p;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// group vtable (one per curve x group)
struct GroupOps {
    int (*buckets)(const void*, const MsmSorted&, MsmScratch&, cudaStream_t, void*, MsmLaunchStats*, cudaStream_t, cudaEvent_t);
    void (*combine)(const uint8_t*, const MsmGeom&, uint8_t*);
    void (*add)(uint8_t*, const uint8_t*);
    void (*to_jacobian)(const uint8_t*, uint8_t*);
    void (*to_affine)(const uint8_t*, uint8_t*);
    void (*from_affine)(const uint8_t*, uint8_t*);
    void (*times)(const uint8_t*, const uint8_t*, int, uint8_t*);
    int (*gen_points)(const uint8_t*, uint64_t, uint64_t, void*, cudaStream_t);
    int (*precompute)(const void*, uint64_t, int, int, void*, cudaStream_t);
    uint32_t xyzz_bytes;
    uint32_t aff_bytes;
};
#define SB_GROUP_OPS(NAME, AFF) GroupOps{NAME##_buckets, NAME##_combine, NAME##_add, NAME##_to_jacobian, NAME##_to_affine, NAME##_from_affine, NAME##_times, NAME##_gen_points, NAME##_precompute, NAME##_xyzz_bytes(), AFF}

struct NttTab { DevBuf lo, hi; int h = 0; };
struct PreTab { DevBuf lo, hi; int h = 0; std::string key; };

struct BaseSet { int group = 0; uint64_t n = 0; void* d = nullptr; void* table = nullptr; MsmGeom gp{}; };

struct Groth16Key {
    uint32_t nVars = 0, nPublic = 0, domainSize = 0; int power = 0;
    std::vector<uint8_t> alpha1, beta1, beta2, gamma2, delta1, delta2;
    void *dA = nullptr, *dB1 = nullptr, *dB2 = nullptr, *dC = nullptr, *dH = nullptr;   // bases (C padded to nVars)
    void *tA = nullptr, *tB1 = nullptr, *tB2 = nullptr, *tC = nullptr, *tH = nullptr;   // precomputed window tables
    MsmGeom gpW{}, gpH{};                                                                // their geometry (precomp != 0 when built)
    // sharded load (multi-GPU): only the point ranges [wlo, wlo+wcnt) of A/B1/B2/C and [hlo, hlo+hcnt) of H are resident
    int shard = 0, n_shards = 1; uint64_t wlo = 0, wcnt = 0, hlo = 0, hcnt = 0;
    uint64_t* d_rowptr = nullptr; uint32_t* d_sig = nullptr; void* d_coef = nullptr; uint64_t nCoef = 0;
    // device work buffers
    bool witness_resident = false;   // set by the first upload: sb_groth16_prove_resident refuses to run before it
    void *dW = nullptr, *dA_T = nullptr, *dB_T = nullptr, *dC_T = nullptr, *dTmp = nullptr, *dTmp2 = nullptr, *dTmp3 = nullptr, *dWsum = nullptr;
};

}  // namespace

namespace { struct PlonkKeyDev; void plonk_free_key(PlonkKeyDev*); }     // api_plonk.inl
namespace { struct FflonkKeyDev; void fflonk_free_key(FflonkKeyDev*); }  // api_fflonk.inl

static constexpr size_t STAGE_BYTES = 8u << 20;

struct sb_ctx {
    // Every entry point that takes a context locks it for the duration of the call: overlapping calls on one context
    // (the reference awaits several bulk calls at once, build/snarkjs.js:14653, 14929-14932; the N-API shim runs them
    // as AsyncWorkers on libuv threads) are serialised here instead of racing on the staging buffers and streams.
    // Recursive because some entries are thin wrappers over others (prove_wtns -> prove, load_file -> load).
    std::recursive_mutex mu;
    int curve = 0, device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint32_t n8q = 32;
    GroupOps g1, g2;
    MsmScratch sort_scratch, bucket_scratch;
    MsmScratch sort_scratch2, bscr[5];           // per-MSM scratch for the overlapped Groth16 pipeline
    cudaStream_t aux[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // high-priority side streams (tails, NTT chain)
    cudaEvent_t pev[16];                         // pipeline events
    uint8_t* pinned = nullptr;                   // 256 KiB pinned staging (window sums, counters)
    uint8_t* stage[2] = {nullptr, nullptr};      // 2 x 8 MiB pinned staging for large pageable host buffers
    cudaEvent_t stage_ev[2];
    MsmLaunchStats stats;
    uint64_t launches = 0;
    DevBuf io[4];
    std::map<int, NttTab> ntt_fwd, ntt_inv;
    DevBuf wr_fwd, wr_inv;
    std::map<int, DevBuf> ninv;           // n^-1 per L
    std::vector<PreTab*> pre_cache;
    std::vector<BaseSet> bases;
    std::vector<Groth16Key*> keys;
    std::vector<PlonkKeyDev*> plonk_keys;
    std::vector<FflonkKeyDev*> fflonk_keys;
    cudaEvent_t ev[8];
    float last_ms[8] = {0};
    int fr_s = 0, fr_bits = 254;
    std::vector<std::vector<uint8_t>> roots;   // w[0..s] Montgomery bytes
    std::vector<uint8_t> nqr, shift;
    std::vector<uint8_t> gen1, gen2;            // affine generators, Montgomery
    cudaEvent_t prof_ev[256];
    double stat[16] = {0};                       // see sb_last_stat
    // multi-GPU (sb_comm_init_rank): one NCCL rank per context
    ncclComm_t comm = nullptr; int rank = 0, world = 1;
    void* d_xchg = nullptr; uint8_t* h_xchg = nullptr;   // partial exchange: world x partial bytes (device / pinned)
};

namespace {

// the message of the last failed call is kept per calling thread, so that two threads sharing a context each read
// their own error text from sb_last_error
thread_local const sb_ctx* t_err_ctx = nullptr;
thread_local std::string t_err;
int fail(sb_ctx* c, int code, const std::string& msg) { if (c) { c->err = msg; t_err_ctx = c; t_err = msg; } return code; }
#define SB_LOCK(c) std::unique_lock<std::recursive_mutex> _sb_lk; if (c) _sb_lk = std::unique_lock<std::recursive_mutex>((c)->mu)
int cuda_fail(sb_ctx* c, cudaError_t e, const char* where) {
    return fail(c, e == cudaErrorMemoryAllocation ? SB_ERR_NOMEM : SB_ERR_CUDA, std::string(where) + ": " + cudaGetErrorString(e));
}
#define CU(c, call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return cuda_fail(c, _e, #call); } while (0)

// Host <-> device copies of caller buffers.  Callers hand us pageable memory (Node Buffers, numpy arrays): the driver's
// own pageable path runs at 5-10 GB/s, so large transfers are staged through two pinned 8 MiB buffers (CPU memcpy of
// chunk k+1 overlaps the DMA of chunk k).  Pinned caller memory (bench.py's witness) and small transfers go direct.
int g_stage_enabled = 1;   // sb_set_tuning(8, 0) falls back to the driver's pageable path
bool host_is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
cudaError_t h2d(sb_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!bytes) return cudaSuccess;
    if (!g_stage_enabled || bytes < (1u << 20) || !c->stage[0] || !c->stage[1] || host_is_pinned(src))
        return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream);
    size_t off = 0; int k = 0; cudaError_t e = cudaSuccess;
    while (off < bytes && e == cudaSuccess) {
        const int b = k & 1; const size_t n = std::min(STAGE_BYTES, bytes - off);
        if (k >= 2) e = cudaEventSynchronize(c->stage_ev[b]);
        if (e != cudaSuccess) break;
        memcpy(c->stage[b], (const uint8_t*)src + off, n);
        e = cudaMemcpyAsync((uint8_t*)dst + off, c->stage[b], n, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaEventRecord(c->stage_ev[b], c->stream);
        off += n; k++;
    }
    // the staging buffers may be reused by the next call: make sure their DMAs are done
    if (e == cudaSuccess) e = cudaEventSynchronize(c->stage_ev[0]);
    if (e == cudaSuccess && k > 1) e = cudaEventSynchronize(c->stage_ev[1]);
    return e;
}
// synchronous on return (the data is in dst)
cudaError_t d2h(sb_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!bytes) return cudaSuccess;
    if (!g_stage_enabled || bytes < (1u << 20) || !c->stage[0] || !c->stage[1] || host_is_pinned(dst)) {
        cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream);
        return e == cudaSuccess ? cudaStreamSynchronize(c->stream) : e;
    }
    size_t off = 0, prev_off = 0, prev_n = 0; int k = 0; cudaError_t e = cudaSuccess;
    while (off < bytes && e == cudaSuccess) {
        const int b = k & 1; const size_t n = std::min(STAGE_BYTES, bytes - off);
        e = cudaMemcpyAsync(c->stage[b], (const uint8_t*)src + off, n, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaEventRecord(c->stage_ev[b], c->stream);
        if (e == cudaSuccess && k >= 1) { e = cudaEventSynchronize(c->stage_ev[b ^ 1]); if (e == cudaSuccess) memcpy((uint8_t*)dst + prev_off, c->stage[b ^ 1], prev_n); }
        prev_off = off; prev_n = n; off += n; k++;
    }
    if (e == cudaSuccess && k >= 1) { const int b = (k - 1) & 1; e = cudaEventSynchronize(c->stage_ev[b]); if (e == cudaSuccess) memcpy((uint8_t*)dst + prev_off, c->stage[b], prev_n); }
    return e;
}

// ------------------------------------------------------------------------------------------------------------
// host Fr helpers, templated on the scalar-field tag
// ------------------------------------------------------------------------------------------------------------
template <class P> struct HostFr {
    typedef Fp<P> F;
    static F from_u32(uint32_t x) { F a = F::zero(); a.v[0] = x; return F::to_mont(a); }
    static void roots(int& s, std::vector<F>& w, F& nqr, F& shift) {
        // reference 12866-12889: nqr = first non-residue from 2, s = 2-adicity, w[s] = nqr^((r-1)/2^s), w[i] = w[i+1]^2
        const int N = P::N;
        uint32_t pm1[N]; for (int i = 0; i < N; i++) pm1[i] = P::p(i); pm1[0] -= 1;
        uint32_t half[N]; for (int i = 0; i < N; i++) half[i] = (pm1[i] >> 1) | (i + 1 < N ? pm1[i + 1] << 31 : 0);
        F negone = F::neg(F::one());
        nqr = from_u32(2);
        while (!(F::pow(nqr, half, N) == negone)) nqr = F::add(nqr, F::one());
        shift = F::sqr(nqr);
        uint32_t t[N]; memcpy(t, pm1, sizeof t); s = 0;
        while (!(t[0] & 1)) { for (int i = 0; i < N; i++) t[i] = (t[i] >> 1) | (i + 1 < N ? t[i + 1] << 31 : 0); s++; }
        w.assign(s + 1, F::zero());
        w[s] = F::pow(nqr, t, N);
        for (int i = s - 1; i >= 0; i--) w[i] = F::sqr(w[i + 1]);
    }
    // lo[e] = base^e (e < 2^h), hi[e] = scale * (base^(2^h))^e (e < nhi)
    static void pow_tables(const F& base, const F& scale, int h, uint64_t nhi, std::vector<F>& lo, std::vector<F>& hi) {
        lo.resize((size_t)1 << h); hi.resize(nhi ? nhi : 1);
        F t = F::one();
        for (size_t e = 0; e < lo.size(); e++) { lo[e] = t; t = F::mul(t, base); }
        F step = t;   // base^(2^h)
        t = scale;
        for (size_t e = 0; e < hi.size(); e++) { hi[e] = t; t = F::mul(t, step); }
    }
};

template <class P> int init_roots(sb_ctx* c) {
    typedef Fp<P> F;
    std::vector<F> w; F nqr, shift; int s;
    HostFr<P>::roots(s, w, nqr, shift);
    c->fr_s = s;
    c->roots.resize(s + 1);
    for (int i = 0; i <= s; i++) c->roots[i].assign((uint8_t*)&w[i], (uint8_t*)&w[i] + 32);
    c->nqr.assign((uint8_t*)&nqr, (uint8_t*)&nqr + 32);
    c->shift.assign((uint8_t*)&shift, (uint8_t*)&shift + 32);
    // in-tile roots w_{2^DMAX}^j and inverse
    F wd = w[NTT_DMAX], wdi = F::inv(wd);
    std::vector<F> lo, hi;
    HostFr<P>::pow_tables(wd, F::one(), NTT_DMAX - 1, 1, lo, hi);
    if (!c->wr_fwd.get(lo.size() * 32)) return SB_ERR_NOMEM;
    cudaMemcpy(c->wr_fwd.p, lo.data(), lo.size() * 32, cudaMemcpyHostToDevice);
    HostFr<P>::pow_tables(wdi, F::one(), NTT_DMAX - 1, 1, lo, hi);
    if (!c->wr_inv.get(lo.size() * 32)) return SB_ERR_NOMEM;
    cudaMemcpy(c->wr_inv.p, lo.data(), lo.size() * 32, cudaMemcpyHostToDevice);
    return 0;
}

template <class P> int build_ntt_tab(sb_ctx* c, int L, bool inverse, NttTab& tab) {
    typedef Fp<P> F;
    F w; memcpy(&w, c->roots[L].data(), 32);
    if (inverse) w = F::inv(w);
    int h = (L + 1) / 2;
    std::vector<F> lo, hi;
    HostFr<P>::pow_tables(w, F::one(), h, (uint64_t)1 << (L - h), lo, hi);
    tab.h = h;
    if (!tab.lo.get(lo.size() * 32) || !tab.hi.get(hi.size() * 32)) return SB_ERR_NOMEM;
    cudaMemcpy(tab.lo.p, lo.data(), lo.size() * 32, cudaMemcpyHostToDevice);
    cudaMemcpy(tab.hi.p, hi.data(), hi.size() * 32, cudaMemcpyHostToDevice);
    return 0;
}

int get_ntt_tab(sb_ctx* c, int L, bool inverse, FrNttTables* out) {
    auto& m = inverse ? c->ntt_inv : c->ntt_fwd;
    auto it = m.find(L);
    if (it == m.end()) {
        NttTab& t = m[L];
        int rc = c->curve == SB_BN254 ? build_ntt_tab<BnFr>(c, L, inverse, t) : build_ntt_tab<BlsFr>(c, L, inverse, t);
        if (rc) { m.erase(L); return fail(c, rc, "ntt table allocation failed"); }
        it = m.find(L);
    }
    out->tw_lo = it->second.lo.p; out->tw_hi = it->second.hi.p; out->h = it->second.h;
    out->wr = inverse ? c->wr_inv.p : c->wr_fwd.p;
    return 0;
}

template <class P> void ninv_bytes(int L, uint8_t* out) {
    typedef Fp<P> F;
    F two = F::add(F::one(), F::one()), n = F::one();
    for (int i = 0; i < L; i++) n = F::mul(n, two);
    F r = F::inv(n); memcpy(out, &r, 32);
}
const void* get_ninv(sb_ctx* c, int L) {
    auto it = c->ninv.find(L);
    if (it == c->ninv.end()) {
        uint8_t b[32];
        if (c->curve == SB_BN254) ninv_bytes<BnFr>(L, b); else ninv_bytes<BlsFr>(L, b);
        DevBuf& d = c->ninv[L];
        if (!d.get(32)) return nullptr;
        cudaMemcpy(d.p, b, 32, cudaMemcpyHostToDevice);
        it = c->ninv.find(L);
    }
    return it->second.p;
}

// apply-key tables for (n, first, inc): lo[e] = inc^e, hi[e] = first * inc^(e 2^h)
template <class P> int build_pre(sb_ctx* c, uint64_t n, const uint8_t* first, const uint8_t* inc, PreTab& t) {
    typedef Fp<P> F;
    int bits = 0; while (((uint64_t)1 << bits) < n) bits++;
    int h = (bits + 1) / 2;
    F f, i; memcpy(&f, first, 32); memcpy(&i, inc, 32);
    std::vector<F> lo, hi;
    HostFr<P>::pow_tables(i, f, h, (n + ((uint64_t)1 << h) - 1) >> h, lo, hi);
    t.h = h;
    if (!t.lo.get(lo.size() * 32) || !t.hi.get(hi.size() * 32)) return SB_ERR_NOMEM;
    cudaMemcpy(t.lo.p, lo.data(), lo.size() * 32, cudaMemcpyHostToDevice);
    cudaMemcpy(t.hi.p, hi.data(), hi.size() * 32, cudaMemcpyHostToDevice);
    return 0;
}
int get_pre(sb_ctx* c, uint64_t n, const uint8_t* first, const uint8_t* inc, FrPre* out) {
    std::string key((const char*)&n, 8); key.append((const char*)first, 32); key.append((const char*)inc, 32);
    for (PreTab* t : c->pre_cache) if (t->key == key) { out->lo = t->lo.p; out->hi = t->hi.p; out->h = t->h; return 0; }
    PreTab* t = new PreTab(); t->key = key;
    int rc = c->curve == SB_BN254 ? build_pre<BnFr>(c, n, first, inc, *t) : build_pre<BlsFr>(c, n, first, inc, *t);
    if (rc) { delete t; return fail(c, rc, "apply-key table allocation failed"); }
    if (c->pre_cache.size() >= 16) { delete c->pre_cache.front(); c->pre_cache.erase(c->pre_cache.begin()); }
    c->pre_cache.push_back(t);
    out->lo = t->lo.p; out->hi = t->hi.p; out->h = t->h;
    return 0;
}

// affine generators as plain big-endian hex (build/snarkjs.js:9468-9472, 9419-9422 region; 10821-10833 for BLS12-381)
template <class P> void hex_to_mont(const char* hex, uint8_t* out) {
    typedef Fp<P> F; F a = F::zero();
    int len = (int)strlen(hex);
    for (int i = 0; i < len; i++) {
        char ch = hex[len - 1 - i];
        uint32_t d = (ch >= '0' && ch <= '9') ? ch - '0' : (ch >= 'a' && ch <= 'f') ? ch - 'a' + 10 : ch - 'A' + 10;
        a.v[i / 8] |= d << (4 * (i % 8));
    }
    a = F::to_mont(a); memcpy(out, &a, sizeof a);
}
void init_generators(sb_ctx* c) {
    if (c->curve == SB_BN254) {
        c->gen1.resize(64); c->gen2.resize(128);
        hex_to_mont<BnFq>("1", c->gen1.data()); hex_to_mont<BnFq>("2", c->gen1.data() + 32);
        hex_to_mont<BnFq>("1800deef121f1e76426a00665e5c4479674322d4f75edadd46debd5cd992f6ed", c->gen2.data());
        hex_to_mont<BnFq>("198e9393920d483a7260bfb731fb5d25f1aa493335a9e71297e485b7aef312c2", c->gen2.data() + 32);
        hex_to_mont<BnFq>("12c85ea5db8c6deb4aab71808dcb408fe3d1e7690c43d37b4ce6cc0166fa7daa", c->gen2.data() + 64);
        hex_to_mont<BnFq>("090689d0585ff075ec9e99ad690c3395bc4b313370b38ef355acdadcd122975b", c->gen2.data() + 96);
    } else {
        c->gen1.resize(96); c->gen2.resize(192);
        hex_to_mont<BlsFq>("17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb", c->gen1.data());
        hex_to_mont<BlsFq>("08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1", c->gen1.data() + 48);
        hex_to_mont<BlsFq>("024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8", c->gen2.data());
        hex_to_mont<BlsFq>("13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e", c->gen2.data() + 48);
        hex_to_mont<BlsFq>("0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801", c->gen2.data() + 96);
        hex_to_mont<BlsFq>("0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be", c->gen2.data() + 144);
    }
}

// profiling helpers: accumulate-kernel event pairs
void prof_begin(sb_ctx* c) { c->stats.ev = c->prof_ev; c->stats.nev = 256; c->stats.used = 0; for (double& d : c->stat) d = 0; }
void prof_end(sb_ctx* c) {
    for (int i = 0; i + 1 < c->stats.used; i += 2) {
        float ms = 0; if (cudaEventElapsedTime(&ms, c->prof_ev[i], c->prof_ev[i + 1]) != cudaSuccess) { cudaGetLastError(); continue; }
        const int g = c->stats.tag[i / 2];
        if (g == PROF_ACC_G1) { c->stat[0] += ms; c->stat[2] += 1; c->stat[9] += ms; }
        else if (g == PROF_ACC_G2) { c->stat[1] += ms; c->stat[3] += 1; c->stat[10] += ms; }
        else if (g == PROF_PAIR_G1) { c->stat[0] += ms; c->stat[9] += ms; }
        else if (g == PROF_PAIR_G2) { c->stat[1] += ms; c->stat[10] += ms; }
        else if (g == PROF_SORT) c->stat[8] += ms;
        else if (g >= PROF_FOLD && g <= PROF_JOIN) c->stat[11 + (g - PROF_FOLD)] += ms;
    }
    c->stats.ev = nullptr; c->stats.used = 0;
}

// Precomputed window tables (msm.cuh k_precompute).  Built for sets of >= 2^12 points whose table index fits the
// 31-bit entry value; g_msm_tuning[3] != 0 disables them (plain windowed Pippenger on the raw bases).
bool want_precomp(sb_ctx* c, uint64_t n) {
    if (g_msm_tuning[3] != 0 || n < (1ull << 12)) return false;
    MsmGeom g = msm_geometry_precomp(n, 32, c->fr_bits);
    return (uint64_t)g.W * n < (1ull << 31);
}
int build_table(sb_ctx* c, const GroupOps& G, const void* d_bases, uint64_t n, void** table, MsmGeom* gp) {
    MsmGeom g = msm_geometry_precomp(n, 32, c->fr_bits);
    cudaError_t e = cudaMalloc(table, (size_t)g.W * n * G.aff_bytes);
    if (e != cudaSuccess) { *table = nullptr; return cuda_fail(c, e, "precompute table allocation"); }
    int rc = G.precompute(d_bases, n, g.c, g.W, *table, c->stream); c->launches++;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "k_precompute");
    e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "k_precompute");
    *gp = g;
    return 0;
}

void tick(sb_ctx* c, int i) { cudaEventRecord(c->ev[i], c->stream); }
float elapsed(sb_ctx* c, int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, c->ev[a], c->ev[b]); return ms; }

// ------------------------------------------------------------------------------------------------------------
// MSM over device-resident bases/scalars: sort once, one bucket pipeline, host recombination.
// acc (host XYZZ bytes) += result
// ------------------------------------------------------------------------------------------------------------
int msm_dev_accumulate(sb_ctx* c, const GroupOps& G, const void* d_bases, const uint8_t* d_scalars, uint32_t sbytes, uint64_t n,
                       uint8_t* acc_xyzz, const MsmGeom* gp = nullptr, uint64_t first = 0) {
    const uint64_t MAXC = 1ull << (g_msm_tuning[6] > 0 ? g_msm_tuning[6] : 23);   // points per MSM chunk (tuning key 6: test hook)
    for (uint64_t off = 0; off < n; off += MAXC) {
        uint64_t cn = std::min(MAXC, n - off);
        MsmGeom g = msm_geometry(cn, sbytes, c->fr_bits);
        if (gp) {   // registered set with precomputed window multiples: d_bases is the table
            g = *gp; g.first = first + off; g.W = (int)((8 * sbytes + 1 + g.c - 1) / g.c);
        }
        MsmSorted s;
        int rc = msm_sort_entries(d_scalars + off * sbytes, sbytes, cn, g, c->sort_scratch, c->stream, &s, &c->stats);
        if (rc) return cuda_fail(c, (cudaError_t)rc, "msm_sort_entries");
        void* d_wsum = c->io[3].get((size_t)g.wsum_points() * G.xyzz_bytes);
        if (!d_wsum) return fail(c, SB_ERR_NOMEM, "out of device memory");
        c->stats.cur_tag = (&G == &c->g1) ? SB_G1 : SB_G2;
        rc = G.buckets(gp ? d_bases : (const void*)((const uint8_t*)d_bases + off * G.aff_bytes), s, c->bucket_scratch, c->stream, d_wsum, &c->stats, nullptr, nullptr);
        if (rc) return cuda_fail(c, (cudaError_t)rc, "msm_buckets");
        std::vector<uint8_t> ws((size_t)g.wsum_points() * G.xyzz_bytes);
        uint64_t entries = 0;
        CU(c, cudaMemcpyAsync(ws.data(), d_wsum, ws.size(), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(&entries, s.counts, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        c->stat[(&G == &c->g1) ? 4 : 5] += (double)entries;
        G.combine(ws.data(), g, acc_xyzz);
    }
    return 0;
}

int msm_host_inputs(sb_ctx* c, int group, const uint8_t* bases, const void* d_bases_opt, const uint8_t* scalars, uint32_t sbytes,
                    uint64_t n, uint8_t* out_jac, uint8_t* out_partial, const MsmGeom* gp = nullptr, uint64_t first = 0) {
    if (!c) return SB_ERR_ARG;
    const GroupOps& G = group == SB_G1 ? c->g1 : c->g2;
    std::vector<uint8_t> acc(G.xyzz_bytes, 0);
    if (n) {
        if (sbytes == 0 || sbytes > 64) return fail(c, SB_ERR_ARG, "Scalar size does not match");
        cudaSetDevice(c->device);
        tick(c, 0);
        const void* d_bases = d_bases_opt;
        if (!d_bases) {
            void* p = c->io[0].get(n * G.aff_bytes);
            if (!p) return fail(c, SB_ERR_NOMEM, "out of device memory");
            CU(c, h2d(c, p, bases, n * G.aff_bytes));
            d_bases = p;
        }
        uint8_t* d_sc = (uint8_t*)c->io[1].get(n * sbytes);
        if (!d_sc) return fail(c, SB_ERR_NOMEM, "out of device memory");
        CU(c, h2d(c, d_sc, scalars, n * sbytes));
        tick(c, 1);
        prof_begin(c);
        int rc = msm_dev_accumulate(c, G, d_bases, d_sc, sbytes, n, acc.data(), gp, first);
        if (rc) return rc;
        tick(c, 2);
        cudaEventSynchronize(c->ev[2]);
        prof_end(c);
        c->last_ms[0] = elapsed(c, 0, 2); c->last_ms[1] = elapsed(c, 0, 1); c->last_ms[2] = elapsed(c, 1, 2);
    }
    if (out_partial) memcpy(out_partial, acc.data(), acc.size());
    if (out_jac) G.to_jacobian(acc.data(), out_jac);
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// binfile / zkey parsing (@iden3/binfileutils readBinFile 17468-17498; src/zkey_utils.js:229-259)
// ------------------------------------------------------------------------------------------------------------
struct Section { uint64_t pos = 0, len = 0; bool present = false; };
int parse_binfile(sb_ctx* c, const uint8_t* d, uint64_t len, const char* magic, uint32_t max_version, std::map<uint32_t, Section>& secs) {
    if (len < 12 || memcmp(d, magic, 4) != 0) return fail(c, SB_ERR_FORMAT, std::string(magic) + ": Invalid File format");
    uint32_t ver, nsec; memcpy(&ver, d + 4, 4); memcpy(&nsec, d + 8, 4);
    if (ver > max_version) return fail(c, SB_ERR_FORMAT, "Version not supported");
    uint64_t pos = 12;
    for (uint32_t i = 0; i < nsec; i++) {
        if (len - pos < 12) return fail(c, SB_ERR_FORMAT, "Invalid file size");
        uint32_t id; uint64_t sl; memcpy(&id, d + pos, 4); memcpy(&sl, d + pos + 4, 8); pos += 12;
        if (sl > len - pos) return fail(c, SB_ERR_FORMAT, "Invalid file size");   // (not pos + sl > len: sl comes from the file and may wrap)
        if (secs[id].present) return fail(c, SB_ERR_FORMAT, "Section Duplicated " + std::to_string(id));
        secs[id].pos = pos; secs[id].len = sl; secs[id].present = true;
        pos += sl;
    }
    if (pos != len) return fail(c, SB_ERR_FORMAT, "Invalid file size");
    return 0;
}

bool modulus_matches(const uint8_t* p, uint32_t n8, int curve, bool scalar_field) {
    uint32_t limbs[12] = {0};
    if (curve == SB_BN254) { if (n8 != 32) return false; for (int i = 0; i < 8; i++) limbs[i] = scalar_field ? BnFr::p(i) : BnFq::p(i); }
    else if (scalar_field) { if (n8 != 32) return false; for (int i = 0; i < 8; i++) limbs[i] = BlsFr::p(i); }
    else { if (n8 != 48) return false; for (int i = 0; i < 12; i++) limbs[i] = BlsFq::p(i); }
    return memcmp(p, limbs, n8) == 0;
}

void free_key(Groth16Key* k) {
    for (void* p : {k->tA, k->tB1, k->tB2, k->tC, k->tH, k->dA, k->dB1, k->dB2, k->dC, k->dH, (void*)k->d_rowptr, (void*)k->d_sig, k->d_coef, k->dW, k->dA_T, k->dB_T, k->dC_T, k->dTmp, k->dTmp2, k->dTmp3, k->dWsum})
        if (p) cudaFree(p);
    delete k;
}

template <class PR> static void fr_from_mont_bytes(const uint8_t* in, uint8_t* out) { Fp<PR> a; memcpy(&a, in, 32); a = Fp<PR>::from_mont(a); memcpy(out, &a, 32); }
template <class PR> static void fr_neg_mul_bytes(const uint8_t* r, const uint8_t* s, uint8_t* out) { Fp<PR> a, b; memcpy(&a, r, 32); memcpy(&b, s, 32); a = Fp<PR>::neg(Fp<PR>::mul(a, b)); memcpy(out, &a, 32); }

}  // namespace

// ================================================================================================================
extern "C" {

const char* sb_version(void) { return "snarkb200 0.2 (sm_100a)"; }
int sb_comm_destroy(sb_ctx* c);

int sb_create(int curve, int device_id, sb_ctx** out) {
    if (!out || (curve != SB_BN254 && curve != SB_BLS12_381)) return SB_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return SB_ERR_NODEVICE;
    if (device_id < 0 || device_id >= ndev) return SB_ERR_ARG;
    if (cudaSetDevice(device_id) != cudaSuccess) return SB_ERR_CUDA;
    sb_ctx* c = new sb_ctx();
    c->curve = curve; c->device = device_id;
    c->n8q = curve == SB_BN254 ? 32 : 48;
    c->fr_bits = curve == SB_BN254 ? 254 : 255;
    if (curve == SB_BN254) { c->g1 = SB_GROUP_OPS(bn254_g1, 64); c->g2 = SB_GROUP_OPS(bn254_g2, 128); }
    else { c->g1 = SB_GROUP_OPS(bls12381_g1, 96); c->g2 = SB_GROUP_OPS(bls12381_g2, 192); }
    if (cudaStreamCreate(&c->stream) != cudaSuccess) { delete c; return SB_ERR_CUDA; }
    for (auto& e : c->ev) cudaEventCreate(&e);
    for (auto& e : c->prof_ev) cudaEventCreate(&e);
    for (auto& e : c->pev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    { int lo = 0, hi = 0; cudaDeviceGetStreamPriorityRange(&lo, &hi);
      for (auto& st : c->aux) cudaStreamCreateWithPriority(&st, cudaStreamDefault, hi); }
    if (cudaHostAlloc((void**)&c->pinned, 256 * 1024, cudaHostAllocDefault) != cudaSuccess) c->pinned = nullptr;
    for (int i = 0; i < 2; i++) { if (cudaHostAlloc((void**)&c->stage[i], STAGE_BYTES, cudaHostAllocDefault) != cudaSuccess) c->stage[i] = nullptr; cudaEventCreateWithFlags(&c->stage_ev[i], cudaEventDisableTiming); }
    init_generators(c);
    int rc = curve == SB_BN254 ? init_roots<BnFr>(c) : init_roots<BlsFr>(c);
    if (rc == 0 && fr_configure(curve) != 0) rc = SB_ERR_CUDA;
    if (rc) { sb_destroy(c); return rc; }
    *out = c;
    return SB_OK;
}

void sb_destroy(sb_ctx* c) {
    if (!c) return;
    sb_comm_destroy(c);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto* k : c->keys) if (k) free_key(k);
    for (auto* k : c->plonk_keys) if (k) plonk_free_key(k);
    for (auto* k : c->fflonk_keys) if (k) fflonk_free_key(k);
    for (auto& b : c->bases) { if (b.d) cudaFree(b.d); if (b.table) cudaFree(b.table); }
    for (auto* t : c->pre_cache) { t->lo.release(); t->hi.release(); delete t; }
    for (auto& kv : c->ntt_fwd) { kv.second.lo.release(); kv.second.hi.release(); }
    for (auto& kv : c->ntt_inv) { kv.second.lo.release(); kv.second.hi.release(); }
    for (auto& kv : c->ninv) kv.second.release();
    c->wr_fwd.release(); c->wr_inv.release();
    for (auto& b : c->io) b.release();
    c->sort_scratch.release(); c->bucket_scratch.release();
    for (auto& e : c->ev) cudaEventDestroy(e);
    for (auto& e : c->prof_ev) cudaEventDestroy(e);
    for (auto& e : c->pev) cudaEventDestroy(e);
    for (auto& st : c->aux) { if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); } }
    if (c->pinned) cudaFreeHost(c->pinned);
    for (int i = 0; i < 2; i++) { if (c->stage[i]) cudaFreeHost(c->stage[i]); cudaEventDestroy(c->stage_ev[i]); }
    c->sort_scratch2.release(); for (auto& b : c->bscr) b.release();
    cudaStreamDestroy(c->stream);
    delete c;
}

const char* sb_last_error(sb_ctx* c) {
    if (!c) return "null context";
    if (t_err_ctx == c) return t_err.c_str();
    SB_LOCK(c); t_err_ctx = c; t_err = c->err; return t_err.c_str();
}
uint64_t sb_launch_count(sb_ctx* c) { SB_LOCK(c); return c ? c->launches + (uint64_t)c->stats.launches : 0; }
float sb_last_ms(sb_ctx* c, int which) { SB_LOCK(c); return (c && which >= 0 && which < 8) ? c->last_ms[which] : 0.f; }
int sb_sync(sb_ctx* c) { SB_LOCK(c); if (!c) return SB_ERR_ARG; cudaSetDevice(c->device); CU(c, cudaStreamSynchronize(c->stream)); return 0; }

int sb_msm_g1_affine(sb_ctx* c, const uint8_t* bases, const uint8_t* scalars, uint32_t sb, uint64_t n, uint8_t* out) { SB_LOCK(c);
    return msm_host_inputs(c, SB_G1, bases, nullptr, scalars, sb, n, out, nullptr);
}
int sb_msm_g2_affine(sb_ctx* c, const uint8_t* bases, const uint8_t* scalars, uint32_t sb, uint64_t n, uint8_t* out) { SB_LOCK(c);
    return msm_host_inputs(c, SB_G2, bases, nullptr, scalars, sb, n, out, nullptr);
}

int sb_bases_register(sb_ctx* c, int group, const uint8_t* bases, uint64_t n, uint64_t* handle) { SB_LOCK(c);
    if (!c || !handle || (group != SB_G1 && group != SB_G2)) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    const GroupOps& G = group == SB_G1 ? c->g1 : c->g2;
    BaseSet b; b.group = group; b.n = n;
    CU(c, cudaMalloc(&b.d, n ? n * G.aff_bytes : 16));
    CU(c, cudaMemcpy(b.d, bases, n * G.aff_bytes, cudaMemcpyHostToDevice));
    if (want_precomp(c, n)) { int rc = build_table(c, G, b.d, n, &b.table, &b.gp); if (rc) { cudaFree(b.d); return rc; } }
    c->bases.push_back(b);
    *handle = c->bases.size();
    return 0;
}
int sb_bases_release(sb_ctx* c, uint64_t h) { SB_LOCK(c);
    if (!c || h == 0 || h > c->bases.size() || !c->bases[h - 1].d) return fail(c, SB_ERR_ARG, "invalid bases handle");
    cudaSetDevice(c->device);
    cudaFree(c->bases[h - 1].d); c->bases[h - 1].d = nullptr; c->bases[h - 1].n = 0;
    if (c->bases[h - 1].table) { cudaFree(c->bases[h - 1].table); c->bases[h - 1].table = nullptr; }
    return 0;
}
static int msm_registered_impl(sb_ctx* c, uint64_t h, uint64_t first, const uint8_t* scalars, uint32_t sb, uint64_t n, uint8_t* out, uint8_t* partial) {
    if (!c || h == 0 || h > c->bases.size() || !c->bases[h - 1].d) return fail(c, SB_ERR_ARG, "invalid bases handle");
    const BaseSet& b = c->bases[h - 1];
    if (first + n > b.n) return fail(c, SB_ERR_ARG, "registered base range out of bounds");
    const GroupOps& G = b.group == SB_G1 ? c->g1 : c->g2;
    if (b.table && sb >= 1 && sb <= 32)
        return msm_host_inputs(c, b.group, nullptr, b.table, scalars, sb, n, out, partial, &b.gp, first);
    return msm_host_inputs(c, b.group, nullptr, (const uint8_t*)b.d + first * G.aff_bytes, scalars, sb, n, out, partial);
}
int sb_msm_registered(sb_ctx* c, uint64_t h, uint64_t first, const uint8_t* scalars, uint32_t sb, uint64_t n, uint8_t* out) { SB_LOCK(c);
    return msm_registered_impl(c, h, first, scalars, sb, n, out, nullptr);
}
int sb_msm_registered_partial(sb_ctx* c, uint64_t h, uint64_t first, const uint8_t* scalars, uint32_t sb, uint64_t n, uint8_t* partial) { SB_LOCK(c);
    return msm_registered_impl(c, h, first, scalars, sb, n, nullptr, partial);
}
uint32_t sb_msm_partial_bytes(sb_ctx* c, int group) { return c ? (group == SB_G1 ? c->g1.xyzz_bytes : c->g2.xyzz_bytes) : 0; }
int sb_msm_sum_partials(sb_ctx* c, int group, const uint8_t* partials, int count, uint8_t* out) { SB_LOCK(c);
    if (!c || (group != SB_G1 && group != SB_G2) || count < 0) return SB_ERR_ARG;
    const GroupOps& G = group == SB_G1 ? c->g1 : c->g2;
    std::vector<uint8_t> acc(G.xyzz_bytes, 0);
    for (int i = 0; i < count; i++) G.add(acc.data(), partials + (size_t)i * G.xyzz_bytes);
    G.to_jacobian(acc.data(), out);
    return 0;
}

int sb_msm_dev(sb_ctx* c, int group, const void* bases_dev, const void* scalars_dev, uint32_t sb, uint64_t n, uint8_t* out) { SB_LOCK(c);
    if (!c || (group != SB_G1 && group != SB_G2)) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    const GroupOps& G = group == SB_G1 ? c->g1 : c->g2;
    std::vector<uint8_t> acc(G.xyzz_bytes, 0);
    tick(c, 0);
    prof_begin(c);
    if (n) { int rc = msm_dev_accumulate(c, G, bases_dev, (const uint8_t*)scalars_dev, sb, n, acc.data()); if (rc) return rc; }
    tick(c, 1); cudaEventSynchronize(c->ev[1]); c->last_ms[0] = elapsed(c, 0, 1);
    prof_end(c);
    G.to_jacobian(acc.data(), out);
    return 0;
}

// ---------------------------------------------------------------------------------------------------- Fr ops
static int ntt_dev(sb_ctx* c, void* a, void* b, uint64_t n, int inverse, const FrPre* pre, bool scale, void** result) {
    if (n == 0 || (n & (n - 1))) return fail(c, SB_ERR_ARG, "fft must be multiple of 2");
    int L = 0; while (((uint64_t)1 << L) < n) L++;
    if (L > c->fr_s) return fail(c, SB_ERR_ARG, "fft size exceeds the 2-adicity of Fr (fftExt path not supported)");
    if (L == 0) { *result = a; return 0; }
    FrNttTables tb;
    int rc = get_ntt_tab(c, L, inverse != 0, &tb); if (rc) return rc;
    const void* post = nullptr;
    if (inverse && scale) { post = get_ninv(c, L); if (!post) return fail(c, SB_ERR_NOMEM, "out of device memory"); }
    int launches = 0;
    ProfScope pn(&c->stats, PROF_NTT, c->stream);
    rc = fr_ntt(c->curve, a, b, L, &tb, pre, post, c->stream, result, &launches);
    pn.end();
    c->launches += launches;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_ntt");
    return 0;
}

int sb_ntt_fr(sb_ctx* c, const uint8_t* in, uint64_t n, int inverse, uint8_t* out) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (n == 0 || (n & (n - 1))) return fail(c, SB_ERR_ARG, "fft must be multiple of 2");
    cudaSetDevice(c->device);
    void* a = c->io[0].get(n * 32); void* b = c->io[1].get(n * 32);
    if (!a || !b) return fail(c, SB_ERR_NOMEM, "out of device memory");
    tick(c, 0);
    CU(c, h2d(c, a, in, n * 32));
    tick(c, 1);
    void* res = nullptr;
    int rc = ntt_dev(c, a, b, n, inverse, nullptr, true, &res); if (rc) return rc;
    tick(c, 2);
    CU(c, d2h(c, out, res, n * 32));
    tick(c, 3);
    CU(c, cudaStreamSynchronize(c->stream));
    c->last_ms[0] = elapsed(c, 0, 3); c->last_ms[1] = elapsed(c, 0, 1); c->last_ms[2] = elapsed(c, 1, 2); c->last_ms[3] = elapsed(c, 2, 3);
    return 0;
}
int sb_ntt_fr_dev(sb_ctx* c, void* data, void* scratch, uint64_t n, int inverse, void** result) { SB_LOCK(c);
    if (!c || !result) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    tick(c, 0);
    int rc = ntt_dev(c, data, scratch, n, inverse, nullptr, true, result); if (rc) return rc;
    tick(c, 1);
    CU(c, cudaStreamSynchronize(c->stream));
    c->last_ms[0] = elapsed(c, 0, 1);
    return 0;
}

int sb_fr_batch_apply_key(sb_ctx* c, const uint8_t* in, uint64_t n, const uint8_t first[32], const uint8_t inc[32], uint8_t* out) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (n == 0) return 0;
    cudaSetDevice(c->device);
    FrPre pre; int rc = get_pre(c, n, first, inc, &pre); if (rc) return rc;
    void* a = c->io[0].get(n * 32); void* b = c->io[1].get(n * 32);
    if (!a || !b) return fail(c, SB_ERR_NOMEM, "out of device memory");
    CU(c, h2d(c, a, in, n * 32));
    rc = fr_apply_key(c->curve, a, b, n, &pre, c->stream); c->launches++;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_apply_key");
    CU(c, d2h(c, out, b, n * 32));
    return 0;
}
static int convert_impl(sb_ctx* c, const uint8_t* in, uint64_t n, uint8_t* out, int to_mont) {
    if (!c) return SB_ERR_ARG;
    if (n == 0) return 0;
    cudaSetDevice(c->device);
    void* a = c->io[0].get(n * 32); void* b = c->io[1].get(n * 32);
    if (!a || !b) return fail(c, SB_ERR_NOMEM, "out of device memory");
    CU(c, h2d(c, a, in, n * 32));
    int rc = fr_convert(c->curve, a, b, n, to_mont, c->stream); c->launches++;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_convert");
    CU(c, d2h(c, out, b, n * 32));
    return 0;
}
int sb_fr_batch_to_montgomery(sb_ctx* c, const uint8_t* in, uint64_t n, uint8_t* out) { SB_LOCK(c); return convert_impl(c, in, n, out, 1); }
int sb_fr_batch_from_montgomery(sb_ctx* c, const uint8_t* in, uint64_t n, uint8_t* out) { SB_LOCK(c); return convert_impl(c, in, n, out, 0); }

int sb_qap_join_abc(sb_ctx* c, const uint8_t* a, const uint8_t* b, const uint8_t* cc, uint64_t n, uint8_t* out) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (n == 0) return 0;
    cudaSetDevice(c->device);
    void* da = c->io[0].get(n * 32); void* db = c->io[1].get(n * 32); void* dc = c->io[2].get(n * 32); void* dout = c->io[3].get(n * 32);
    if (!da || !db || !dc || !dout) return fail(c, SB_ERR_NOMEM, "out of device memory");
    CU(c, h2d(c, da, a, n * 32));
    CU(c, h2d(c, db, b, n * 32));
    CU(c, h2d(c, dc, cc, n * 32));
    int rc = fr_join_abc(c->curve, da, db, dc, dout, n, c->stream); c->launches++;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_join_abc");
    CU(c, d2h(c, out, dout, n * 32));
    return 0;
}

int sb_fr_root(sb_ctx* c, int what, uint8_t out[32]) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (what == -1) memcpy(out, c->shift.data(), 32);
    else if (what == -2) memcpy(out, c->nqr.data(), 32);
    else if (what >= 0 && what <= c->fr_s) memcpy(out, c->roots[what].data(), 32);
    else return fail(c, SB_ERR_ARG, "root index out of range");
    return c->fr_s;
}

int sb_set_tuning(int key, int value) {
    if (key == 8) { g_stage_enabled = value; return 0; }                                                      // pinned staging of pageable buffers
    if (key == 7) { if (value < 10 || value > 12) return SB_ERR_ARG; g_ntt_tile_log = value; return 0; }   // NTT tile size
    if (key == 9) { g_msm_tuning[7] = value; return 0; }                                                      // forced entries per accumulation thread (0 = adaptive)
    if (key == 12) { g_msm_tuning[10] = value; return 0; }                                                    // minBlocksPerSM variant of the 8-limb base-field accumulation (BN254 G1): 4 default, 3, 2
    if (key == 11) { g_msm_tuning[9] = value; return 0; }                                                     // lane-pair G2 accumulation (k_accumulate_pair): 0 = off, 3 / 4 = minBlocksPerSM
    if (key == 10) { g_msm_tuning[8] = value; return 0; }                                                     // minBlocksPerSM variant of the 12-limb base-field accumulation (BLS12-381 G1)
    if (key < 0 || key >= 7) return SB_ERR_ARG; g_msm_tuning[key] = value; return 0;
}
double sb_last_stat(sb_ctx* c, int which) { SB_LOCK(c); return (c && which >= 0 && which < 16) ? c->stat[which] : 0.0; }
double sb_calibrate(sb_ctx* c, int what) { SB_LOCK(c); if (!c) return -1; cudaSetDevice(c->device); return calibrate(what, c->stream); }
int sb_gen_points(sb_ctx* c, int group, uint64_t seed, uint64_t n, uint8_t* out) { SB_LOCK(c);
    if (!c || (group != SB_G1 && group != SB_G2)) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    const GroupOps& G = group == SB_G1 ? c->g1 : c->g2;
    void* d = c->io[0].get(n * G.aff_bytes);
    if (!d) return fail(c, SB_ERR_NOMEM, "out of device memory");
    int rc = G.gen_points(group == SB_G1 ? c->gen1.data() : c->gen2.data(), seed, n, d, c->stream); c->launches++;
    if (rc) return cuda_fail(c, (cudaError_t)rc, "gen_points");
    CU(c, d2h(c, out, d, n * G.aff_bytes));
    return 0;
}
int sb_generator(sb_ctx* c, int group, uint8_t* out) { SB_LOCK(c);
    if (!c || (group != SB_G1 && group != SB_G2)) return SB_ERR_ARG;
    const std::vector<uint8_t>& g = group == SB_G1 ? c->gen1 : c->gen2;
    memcpy(out, g.data(), g.size()); return 0;
}

void* sb_dev_alloc(sb_ctx* c, uint64_t bytes) { SB_LOCK(c); if (!c) return nullptr; cudaSetDevice(c->device); void* p = nullptr; if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr; return p; }
int sb_dev_free(sb_ctx* c, void* p) { SB_LOCK(c); if (!c) return SB_ERR_ARG; cudaSetDevice(c->device); CU(c, cudaFree(p)); return 0; }
int sb_dev_upload(sb_ctx* c, void* dst, const uint8_t* src, uint64_t bytes) { SB_LOCK(c); if (!c) return SB_ERR_ARG; cudaSetDevice(c->device); CU(c, h2d(c, dst, src, bytes)); CU(c, cudaStreamSynchronize(c->stream)); return 0; }
int sb_dev_download(sb_ctx* c, uint8_t* dst, const void* src, uint64_t bytes) { SB_LOCK(c); if (!c) return SB_ERR_ARG; cudaSetDevice(c->device); CU(c, d2h(c, dst, src, bytes)); return 0; }

// ---------------------------------------------------------------------------------------------------- Groth16
// A zkey comes either as a memory image (z != nullptr) or as a file streamed section by section: the small sections
// (1, 2, 4) are read to the host, the base sections (5-9) go straight to HBM through two pinned staging buffers with
// cudaMemcpyAsync overlapping the next fread (SURVEY §8f rank 2).
struct ZkeySource {
    const uint8_t* z = nullptr; uint64_t zlen = 0; FILE* f = nullptr;
    std::vector<uint8_t> small[5];   // host copies of sections 1, 2, 4 when streaming
};
static int zkey_section_table(sb_ctx* c, ZkeySource& src, std::map<uint32_t, Section>& secs) {
    if (src.z) return parse_binfile(c, src.z, src.zlen, "zkey", 2, secs);
    uint8_t hd[12];
    if (fseek(src.f, 0, SEEK_END)) return fail(c, SB_ERR_FORMAT, "zkey: seek failed");
    const uint64_t flen = (uint64_t)ftell(src.f);
    fseek(src.f, 0, SEEK_SET);
    if (fread(hd, 1, 12, src.f) != 12 || memcmp(hd, "zkey", 4) != 0) return fail(c, SB_ERR_FORMAT, "zkey: Invalid File format");
    uint32_t ver, nsec; memcpy(&ver, hd + 4, 4); memcpy(&nsec, hd + 8, 4);
    if (ver > 2) return fail(c, SB_ERR_FORMAT, "Version not supported");
    uint64_t pos = 12;
    for (uint32_t i = 0; i < nsec; i++) {
        if (fseek(src.f, (long)pos, SEEK_SET) || fread(hd, 1, 12, src.f) != 12) return fail(c, SB_ERR_FORMAT, "Invalid file size");
        uint32_t id; uint64_t sl; memcpy(&id, hd, 4); memcpy(&sl, hd + 4, 8); pos += 12;
        if (pos > flen || sl > flen - pos) return fail(c, SB_ERR_FORMAT, "Invalid file size");
        if (secs[id].present) return fail(c, SB_ERR_FORMAT, "Section Duplicated " + std::to_string(id));
        secs[id].pos = pos; secs[id].len = sl; secs[id].present = true; pos += sl;
    }
    if (pos != flen) return fail(c, SB_ERR_FORMAT, "Invalid file size");
    return 0;
}
// host pointer to a small section
static const uint8_t* zkey_host_section(ZkeySource& src, const std::map<uint32_t, Section>& secs, uint32_t id, int slot) {
    const Section& s = secs.at(id);
    if (src.z) return src.z + s.pos;
    src.small[slot].resize(s.len ? s.len : 1);
    if (fseek(src.f, (long)s.pos, SEEK_SET) || fread(src.small[slot].data(), 1, s.len, src.f) != s.len) return nullptr;
    return src.small[slot].data();
}
// section bytes [off, off+len) -> device
static cudaError_t zkey_to_device(sb_ctx* c, ZkeySource& src, const std::map<uint32_t, Section>& secs, uint32_t id, uint64_t off, uint64_t len, void* dst) {
    if (!len) return cudaSuccess;
    const Section& s = secs.at(id);
    if (src.z) return cudaMemcpy(dst, src.z + s.pos + off, len, cudaMemcpyHostToDevice);
    const size_t CH = 16u << 20;
    uint8_t* pin[2] = {nullptr, nullptr}; cudaEvent_t ev[2];
    cudaError_t e = cudaHostAlloc((void**)&pin[0], CH, cudaHostAllocDefault); if (e != cudaSuccess) return e;
    e = cudaHostAlloc((void**)&pin[1], CH, cudaHostAllocDefault); if (e != cudaSuccess) { cudaFreeHost(pin[0]); return e; }
    cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming); cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
    if (fseek(src.f, (long)(s.pos + off), SEEK_SET)) e = cudaErrorUnknown;
    uint64_t done = 0; int b = 0; bool used[2] = {false, false};
    while (e == cudaSuccess && done < len) {
        const size_t n = (size_t)std::min<uint64_t>(CH, len - done);
        if (used[b]) e = cudaEventSynchronize(ev[b]);                   // staging buffer free again?
        if (e == cudaSuccess && fread(pin[b], 1, n, src.f) != n) e = cudaErrorUnknown;
        if (e == cudaSuccess) e = cudaMemcpyAsync((uint8_t*)dst + done, pin[b], n, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) { cudaEventRecord(ev[b], c->stream); used[b] = true; }
        done += n; b ^= 1;
    }
    cudaStreamSynchronize(c->stream);
    cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]); cudaFreeHost(pin[0]); cudaFreeHost(pin[1]);
    return e;
}

static int groth16_load_impl(sb_ctx* c, ZkeySource& src, int shard, int n_shards, uint64_t* handle) {
    if (!c || (!src.z && !src.f) || !handle || n_shards < 1 || shard < 0 || shard >= n_shards) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    std::map<uint32_t, Section> secs;
    int rc = zkey_section_table(c, src, secs); if (rc) return rc;
    for (uint32_t id : {1u, 2u, 4u, 5u, 6u, 7u, 8u, 9u}) if (!secs[id].present) return fail(c, SB_ERR_FORMAT, "Missing section " + std::to_string(id));
    const uint8_t* s1 = zkey_host_section(src, secs, 1, 0);
    if (!s1 || secs[1].len < 4) return fail(c, SB_ERR_FORMAT, "zkey: short read");
    uint32_t proto; memcpy(&proto, s1, 4);
    if (proto != 1) return fail(c, SB_ERR_FORMAT, "zkey file is not groth16");
    const uint8_t* h = zkey_host_section(src, secs, 2, 1); uint64_t hl = secs[2].len;
    if (!h) return fail(c, SB_ERR_FORMAT, "zkey: short read");
    const uint32_t n8q = c->n8q, n8r = 32;
    const uint64_t need = 4 + n8q + 4 + n8r + 12 + 3 * 2 * n8q + 3 * 4 * n8q;
    if (hl < need) return fail(c, SB_ERR_FORMAT, "zkey header too short");
    uint32_t v; memcpy(&v, h, 4);
    if (v != n8q || !modulus_matches(h + 4, n8q, c->curve, false)) return fail(c, SB_ERR_FORMAT, "zkey curve does not match the context curve");
    memcpy(&v, h + 4 + n8q, 4);
    if (v != n8r || !modulus_matches(h + 8 + n8q, n8r, c->curve, true)) return fail(c, SB_ERR_FORMAT, "zkey curve does not match the context curve");
    Groth16Key* k = new Groth16Key();
    const uint8_t* q = h + 8 + n8q + n8r;
    memcpy(&k->nVars, q, 4); memcpy(&k->nPublic, q + 4, 4); memcpy(&k->domainSize, q + 8, 4); q += 12;
    const uint32_t sG1 = 2 * n8q, sG2 = 4 * n8q;
    k->alpha1.assign(q, q + sG1); q += sG1; k->beta1.assign(q, q + sG1); q += sG1;
    k->beta2.assign(q, q + sG2); q += sG2; k->gamma2.assign(q, q + sG2); q += sG2;
    k->delta1.assign(q, q + sG1); q += sG1; k->delta2.assign(q, q + sG2);
    const uint64_t n = k->domainSize, nv = k->nVars;
    if (n == 0 || (n & (n - 1))) { delete k; return fail(c, SB_ERR_FORMAT, "domain size is not a power of two"); }
    while (((uint64_t)1 << k->power) < n) k->power++;
    if (k->power > c->fr_s) { delete k; return fail(c, SB_ERR_FORMAT, "Circuit too big for this curve"); }
    if (nv < (uint64_t)k->nPublic + 1) { delete k; return fail(c, SB_ERR_FORMAT, "invalid zkey header"); }
    if (secs[5].len != nv * sG1 || secs[6].len != nv * sG1 || secs[7].len != nv * sG2 ||
        secs[8].len != (nv - k->nPublic - 1) * sG1 || secs[9].len != n * sG1) { delete k; return fail(c, SB_ERR_FORMAT, "zkey section size mismatch"); }
    // coefficient section -> CSR over rows (matrix m, constraint c): src/zkey_utils.js:110-118, groth16_prove.js:147-187
    const uint8_t* s4 = zkey_host_section(src, secs, 4, 2);
    if (!s4 || secs[4].len < 4) { delete k; return fail(c, SB_ERR_FORMAT, "zkey: short read"); }
    uint32_t ncoef; memcpy(&ncoef, s4, 4);
    const uint64_t sCoef = 12 + n8r;
    if (secs[4].len != 4 + ncoef * sCoef) { delete k; return fail(c, SB_ERR_FORMAT, "zkey coefficient section size mismatch"); }
    const uint8_t* cf = s4 + 4;
    std::vector<uint64_t> rowptr(2 * n + 1, 0);
    for (uint64_t i = 0; i < ncoef; i++) {
        uint32_t m, cc, s; memcpy(&m, cf + i * sCoef, 4); memcpy(&cc, cf + i * sCoef + 4, 4); memcpy(&s, cf + i * sCoef + 8, 4);
        if (m > 1 || cc >= n || s >= nv) { delete k; return fail(c, SB_ERR_FORMAT, "zkey coefficient out of range"); }
        rowptr[m * n + cc + 1]++;
    }
    for (uint64_t i = 0; i < 2 * n; i++) rowptr[i + 1] += rowptr[i];
    std::vector<uint64_t> cursor(rowptr.begin(), rowptr.end() - 1);
    std::vector<uint32_t> sig(ncoef ? ncoef : 1); std::vector<uint8_t> coef((size_t)(ncoef ? ncoef : 1) * 32);
    for (uint64_t i = 0; i < ncoef; i++) {
        uint32_t m, cc, s; memcpy(&m, cf + i * sCoef, 4); memcpy(&cc, cf + i * sCoef + 4, 4); memcpy(&s, cf + i * sCoef + 8, 4);
        uint64_t p = cursor[m * n + cc]++;
        sig[p] = s; memcpy(&coef[p * 32], cf + i * sCoef + 12, 32);
    }
    k->nCoef = ncoef;
    cudaError_t e = cudaSuccess;
    auto up = [&](void** d, const void* src, size_t bytes, size_t alloc) {
        if (e != cudaSuccess) return;
        e = cudaMalloc(d, alloc ? alloc : 16); if (e != cudaSuccess) return;
        if (bytes) e = cudaMemcpy(*d, src, bytes, cudaMemcpyHostToDevice);
    };
    k->shard = shard; k->n_shards = n_shards;
    sb_shard_range(nv, shard, n_shards, &k->wlo, &k->wcnt);
    sb_shard_range(n, shard, n_shards, &k->hlo, &k->hcnt);
    const uint64_t wlo = k->wlo, wcnt = k->wcnt, hlo = k->hlo, hcnt = k->hcnt;
    auto upsec = [&](void** d, uint32_t id, uint64_t off, uint64_t len) {
        if (e != cudaSuccess) return;
        e = cudaMalloc(d, len ? len : 16); if (e != cudaSuccess) return;
        e = zkey_to_device(c, src, secs, id, off, len, *d);
    };
    upsec(&k->dA, 5, wlo * sG1, wcnt * sG1);
    upsec(&k->dB1, 6, wlo * sG1, wcnt * sG1);
    upsec(&k->dB2, 7, wlo * sG2, wcnt * sG2);
    // C bases are indexed by signal - (nPublic+1): pad so that one sorted digit list of the witness serves A, B1, B2 and C
    if (e == cudaSuccess) {
        const uint64_t np1 = (uint64_t)k->nPublic + 1;
        e = cudaMalloc(&k->dC, wcnt ? wcnt * sG1 : 16);
        if (e == cudaSuccess && wcnt) e = cudaMemset(k->dC, 0, wcnt * sG1);
        const uint64_t g0 = std::max(wlo, np1), g1 = wlo + wcnt;
        if (e == cudaSuccess && g1 > g0) e = zkey_to_device(c, src, secs, 8, (g0 - np1) * sG1, (g1 - g0) * sG1, (uint8_t*)k->dC + (g0 - wlo) * sG1);
    }
    upsec(&k->dH, 9, hlo * sG1, hcnt * sG1);
    up((void**)&k->d_rowptr, rowptr.data(), rowptr.size() * 8, rowptr.size() * 8);
    up((void**)&k->d_sig, sig.data(), (size_t)ncoef * 4, (size_t)ncoef * 4);
    up(&k->d_coef, coef.data(), (size_t)ncoef * 32, (size_t)ncoef * 32);
    up(&k->dW, nullptr, 0, (nv + 64) * 32);   // + room for the padded slices of the distributed witness all-gather
    up(&k->dA_T, nullptr, 0, n * 32); up(&k->dB_T, nullptr, 0, n * 32); up(&k->dC_T, nullptr, 0, n * 32); up(&k->dTmp, nullptr, 0, n * 32);
    up(&k->dTmp2, nullptr, 0, n * 32); up(&k->dTmp3, nullptr, 0, n * 32);
    up(&k->dWsum, nullptr, 0, 8 * 80 * 4 * 96);
    if (e != cudaSuccess) { free_key(k); return cuda_fail(c, e, "sb_groth16_load upload"); }
    if (want_precomp(c, wcnt) && want_precomp(c, hcnt)) {
        int rc2 = build_table(c, c->g1, k->dA, wcnt, &k->tA, &k->gpW);
        if (!rc2) rc2 = build_table(c, c->g1, k->dB1, wcnt, &k->tB1, &k->gpW);
        if (!rc2) rc2 = build_table(c, c->g2, k->dB2, wcnt, &k->tB2, &k->gpW);
        if (!rc2) rc2 = build_table(c, c->g1, k->dC, wcnt, &k->tC, &k->gpW);
        if (!rc2) rc2 = build_table(c, c->g1, k->dH, hcnt, &k->tH, &k->gpH);
        if (rc2) { free_key(k); return rc2; }
    }
    c->keys.push_back(k);
    *handle = c->keys.size();
    return 0;
}

int sb_groth16_load(sb_ctx* c, const uint8_t* z, uint64_t zlen, uint64_t* handle) { SB_LOCK(c);
    if (!z) return SB_ERR_ARG;
    ZkeySource src; src.z = z; src.zlen = zlen; return groth16_load_impl(c, src, 0, 1, handle);
}
int sb_groth16_load_sharded(sb_ctx* c, const uint8_t* z, uint64_t zlen, int shard, int n_shards, uint64_t* handle) { SB_LOCK(c);
    if (!z) return SB_ERR_ARG;
    ZkeySource src; src.z = z; src.zlen = zlen; return groth16_load_impl(c, src, shard, n_shards, handle);
}

int sb_groth16_load_file(sb_ctx* c, const char* path, uint64_t* handle) { SB_LOCK(c);
    if (!c || !path) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, SB_ERR_FORMAT, std::string("cannot open ") + path);
    ZkeySource src; src.f = f;
    int rc = groth16_load_impl(c, src, 0, 1, handle);
    fclose(f);
    return rc;
}

static Groth16Key* get_key(sb_ctx* c, uint64_t h) { return (c && h >= 1 && h <= c->keys.size()) ? c->keys[h - 1] : nullptr; }

int sb_groth16_info(sb_ctx* c, uint64_t h, uint32_t* nv, uint32_t* np, uint32_t* ds) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    if (nv) *nv = k->nVars; if (np) *np = k->nPublic; if (ds) *ds = k->domainSize;
    return 0;
}
int sb_groth16_release(sb_ctx* c, uint64_t h) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    cudaSetDevice(c->device); free_key(k); c->keys[h - 1] = nullptr; return 0;
}
uint32_t sb_groth16_partials_bytes(sb_ctx* c) { return c ? 4 * c->g1.xyzz_bytes + c->g2.xyzz_bytes : 0; }

// ---------------------------------------------------------------------------------------------------- NCCL
// libnccl is opened on first use, so libsnarkb200.so loads (and every single-GPU entry works) on hosts without NCCL.
// If the process already has a libnccl.so.2 (torch bundles one) that copy is reused.
struct NcclApi {
    void* so = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi* nccl_api(std::string* why) {
    static std::mutex mu; static NcclApi api; static bool tried = false; static std::string err;
    std::lock_guard<std::mutex> lk(mu);
    if (!tried) {
        tried = true;
        const char* env = getenv("SB_NCCL_LIB");
        void* so = env ? dlopen(env, RTLD_NOW | RTLD_LOCAL) : nullptr;
        if (!so) so = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (!so) so = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!so) so = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
        if (!so) err = std::string("cannot load libnccl.so.2: ") + dlerror();
        else {
            api.so = so;
            bool ok = true;
            auto sym = [&](const char* n) { void* p = dlsym(so, n); if (!p) { ok = false; err = std::string("libnccl: missing symbol ") + n; } return p; };
            api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
            api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
            api.Send = (decltype(api.Send))sym("ncclSend");
            api.Recv = (decltype(api.Recv))sym("ncclRecv");
            api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
            api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
            api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
            if (!ok) api.so = nullptr;
        }
    }
    if (!api.so) { if (why) *why = err; return nullptr; }
    return &api;
}
#define NC(c, api, call) do { ncclResult_t _r = (call); if (_r != ncclSuccess) return fail(c, SB_ERR_CUDA, std::string(#call) + ": " + (api)->GetErrorString(_r)); } while (0)

int sb_comm_unique_id(uint8_t out[128]) {
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    if (!out) return SB_ERR_ARG;
    NcclApi* nc = nccl_api(nullptr); if (!nc) return SB_ERR_CUDA;
    ncclUniqueId id; if (nc->GetUniqueId(&id) != ncclSuccess) return SB_ERR_CUDA;
    memcpy(out, &id, 128); return 0;
}
int sb_comm_init_rank(sb_ctx* c, int world, int rank, const uint8_t id_bytes[128]) { SB_LOCK(c);
    if (!c || !id_bytes || world < 1 || world > 64 || rank < 0 || rank >= world) return fail(c, SB_ERR_ARG, "invalid communicator arguments");
    if (c->comm) return fail(c, SB_ERR_ARG, "context already belongs to a communicator");
    std::string why; NcclApi* nc = nccl_api(&why); if (!nc) return fail(c, SB_ERR_CUDA, why);
    cudaSetDevice(c->device);
    ncclUniqueId id; memcpy(&id, id_bytes, 128);
    NC(c, nc, nc->CommInitRank(&c->comm, world, id, rank));
    c->rank = rank; c->world = world;
    const size_t pb = (size_t)sb_groth16_partials_bytes(c);
    CU(c, cudaMalloc(&c->d_xchg, pb * world));
    CU(c, cudaHostAlloc((void**)&c->h_xchg, pb * (world + 1), cudaHostAllocDefault));
    return 0;
}
int sb_comm_info(sb_ctx* c, int* rank, int* world) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (rank) *rank = c->rank; if (world) *world = c->comm ? c->world : 0;
    return 0;
}
int sb_comm_destroy(sb_ctx* c) { SB_LOCK(c);
    if (!c) return SB_ERR_ARG;
    if (c->comm) {
        cudaSetDevice(c->device); cudaStreamSynchronize(c->stream);
        if (NcclApi* nc = nccl_api(nullptr)) nc->CommDestroy(c->comm);
        c->comm = nullptr; c->rank = 0; c->world = 1;
        if (c->d_xchg) cudaFree(c->d_xchg); if (c->h_xchg) cudaFreeHost(c->h_xchg);
        c->d_xchg = nullptr; c->h_xchg = nullptr;
    }
    return 0;
}
// which rank runs the iNTT -> coset NTT chain of polynomial j (0 = A, 1 = B, 2 = C) when a proof is distributed
int sb_dist_chain_owner(int chain, int world) { return world > 0 ? chain % world : 0; }

// plain (non-Montgomery) r and s: when given, the prover folds s*A + r*B1 + H into the C partial as soon as A and B1 land
// (hidden behind the C and H MSMs), so that the proof assembly after the last MSM is three additions
struct ProofScalars { uint8_t rp[32], sp[32]; };

// device part of the prover: returns the five MSM partials (A, B1, C, H | B2) as host XYZZ bytes.
// dist: this context is rank c->rank of c->world (sb_comm_init_rank); the witness is uploaded in slices and all-gathered,
// the three transform chains run on different ranks and exchange their coset evaluations (NCCL send/recv), every rank
// then joins and multiplies its own H range.
static int groth16_device(sb_ctx* c, Groth16Key* k, const uint8_t* witness, uint64_t n_witness, int shard, int n_shards, uint8_t* partials,
                          const ProofScalars* ps = nullptr, bool dist = false) {
    if (witness && n_witness != k->nVars) return fail(c, SB_ERR_ARG, "Invalid witness length. Circuit: " + std::to_string(k->nVars) + ", witness: " + std::to_string(n_witness));
    cudaSetDevice(c->device);
    const uint64_t n = k->domainSize, nv = k->nVars;
    const int cv = c->curve;
    NcclApi* nc = nullptr;
    if (dist) {
        if (!c->comm) return fail(c, SB_ERR_ARG, "context has no communicator: call sb_comm_init_rank first");
        nc = nccl_api(nullptr);
        shard = c->rank; n_shards = c->world;
    }
    const int world = n_shards, rank = shard;
    int rc;
    tick(c, 0);
    if (witness) {
        k->witness_resident = false;
        if (dist && world > 1) {   // every rank uploads 1/world of the witness; NVLink all-gather completes it
            const uint64_t per = (nv + world - 1) / world, lo = std::min(nv, per * (uint64_t)rank), cnt = std::min(nv - lo, per);
            CU(c, h2d(c, (uint8_t*)k->dW + lo * 32, witness + lo * 32, cnt * 32));
            NC(c, nc, nc->AllGather((const uint8_t*)k->dW + per * rank * 32, k->dW, per * 32, ncclUint8, c->comm, c->stream));
        } else CU(c, h2d(c, k->dW, witness, nv * 32));
        k->witness_resident = true;
    } else if (!k->witness_resident) return fail(c, SB_ERR_ARG, "no witness resident for this proving key: call sb_groth16_prove first");
    tick(c, 1);
    prof_begin(c);
    // MSMs (:84-101).  Shard = contiguous point range (SURVEY §8e); shard 0 of 1 = everything.
    auto range_of = [&](uint64_t total, int sh, uint64_t& lo, uint64_t& cnt) { sb_shard_range(total, sh, n_shards, &lo, &cnt); };
    uint64_t wlo, wcnt; range_of(nv, rank, wlo, wcnt);
    uint64_t hlo, hcnt; range_of(n, rank, hlo, hcnt);
    // chain j (0 = A, 1 = B, 2 = C) runs on rank owner(j); without a communicator every chain runs here
    auto owner = [&](int j) { return (dist && world > 1) ? sb_dist_chain_owner(j, world) : rank; };
    void* bufs[3] = {k->dA_T, k->dB_T, k->dC_T}; void* scr[3] = {k->dTmp, k->dTmp2, k->dTmp3};
    // where the chain results end up depends only on the pass count: known on ranks that run no chain too
    const int np = fr_ntt_passes(k->power);
    void* odd[3]; void* tmp;
    { const bool x_scr = (np & 1) != 0;                          // after the inverse transform the data sits in scr iff np is odd
      for (int j = 0; j < 3; j++) { void* X = x_scr ? scr[j] : bufs[j]; void* Y = x_scr ? bufs[j] : scr[j]; odd[j] = (np & 1) ? Y : X; }
      tmp = (odd[0] == bufs[0]) ? scr[0] : bufs[0]; }
    auto run_qap_ntt = [&]() -> int {
        int my[3], m = 0;
        for (int j = 0; j < 3; j++) if (owner(j) == rank) my[m++] = j;
        if (m) {
            // buildABC1 (:147-187)
            { ProfScope pq(&c->stats, PROF_QAP, c->stream);
              rc = fr_qap_rows(cv, k->d_rowptr, k->d_sig, k->d_coef, k->dW, k->dA_T, k->dB_T, k->dC_T, n, c->stream); c->launches++;
              pq.end(); }
            if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_qap_rows");
            // :64-76  ifft -> batchApplyKey(1, inc) -> fft, with 1/n of the inverse folded into the coset table
            const uint8_t* inc = (k->power == c->fr_s) ? c->shift.data() : c->roots[k->power + 1].data();
            uint8_t ninv[32];
            if (cv == SB_BN254) ninv_bytes<BnFr>(k->power, ninv); else ninv_bytes<BlsFr>(k->power, ninv);
            FrPre pre; rc = get_pre(c, n, ninv, inc, &pre); if (rc) return rc;
            // this rank's transforms run as one batch per pass (grids fill whole waves)
            void* a[3]; void* b[3];
            for (int i = 0; i < m; i++) { a[i] = bufs[my[i]]; b[i] = scr[my[i]]; }
            FrNttTables tbi, tbf;
            rc = get_ntt_tab(c, k->power, true, &tbi); if (rc) return rc;
            rc = get_ntt_tab(c, k->power, false, &tbf); if (rc) return rc;
            int side = 0, launches = 0;
            ProfScope pn(&c->stats, PROF_NTT, c->stream);
            rc = fr_ntt_batch(cv, a, b, m, k->power, &tbi, nullptr, nullptr, c->stream, &side, &launches);      // unscaled inverse
            if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_ntt_batch");
            void** src = side ? b : a; void** dst = side ? a : b;
            int side2 = 0;
            rc = fr_ntt_batch(cv, src, dst, m, k->power, &tbf, &pre, nullptr, c->stream, &side2, &launches);     // coset NTT, 1/n folded in
            if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_ntt_batch");
            pn.end();
            c->launches += launches;
            void** res = side2 ? dst : src;
            for (int i = 0; i < m; i++) if (res[i] != odd[my[i]]) return fail(c, SB_ERR_CUDA, "internal: NTT result buffer mismatch");
        }
        if (dist && world > 1) {   // coset evaluations of chain j: owner -> every other rank's H range
            NC(c, nc, nc->GroupStart());
            for (int j = 0; j < 3; j++) {
                const int o = owner(j);
                if (o == rank) {
                    for (int q = 0; q < world; q++) {
                        if (q == rank) continue;
                        uint64_t qlo, qcnt; range_of(n, q, qlo, qcnt);
                        if (qcnt) NC(c, nc, nc->Send((const uint8_t*)odd[j] + qlo * 32, qcnt * 32, ncclUint8, q, c->comm, c->stream));
                    }
                } else if (hcnt) NC(c, nc, nc->Recv((uint8_t*)odd[j] + hlo * 32, hcnt * 32, ncclUint8, o, c->comm, c->stream));
            }
            NC(c, nc, nc->GroupEnd());
        }
        // joinABC (:320-374) -> plain scalars for the H MSM, over this rank's H range, into the remaining scratch buffer
        if (hcnt) {
            ProfScope pj(&c->stats, PROF_JOIN, c->stream);
            rc = fr_join_abc(cv, (const uint8_t*)odd[0] + hlo * 32, (const uint8_t*)odd[1] + hlo * 32, (const uint8_t*)odd[2] + hlo * 32,
                             (uint8_t*)tmp + hlo * 32, hcnt, c->stream); c->launches++;
            pj.end();
            if (rc) return cuda_fail(c, (cudaError_t)rc, "fr_join_abc");
        }
        return 0;
    };
    const GroupOps& G1 = c->g1; const GroupOps& G2 = c->g2;
    uint8_t* pA = partials; uint8_t* pB1 = pA + G1.xyzz_bytes; uint8_t* pC = pB1 + G1.xyzz_bytes; uint8_t* pH = pC + G1.xyzz_bytes; uint8_t* pB2 = pH + G1.xyzz_bytes;
    memset(partials, 0, 4 * G1.xyzz_bytes + G2.xyzz_bytes);
    std::vector<uint8_t> sA(G1.xyzz_bytes, 0), rB1(G1.xyzz_bytes, 0);
    const uint64_t MAXC = 1ull << (g_msm_tuning[6] > 0 ? g_msm_tuning[6] : 23);   // points per MSM chunk (tuning key 6: test hook)
    // a key loaded with sb_groth16_load_sharded only holds its own ranges: local indexing
    const bool local = k->n_shards > 1;
    if (local && (shard != k->shard || n_shards != k->n_shards)) return fail(c, SB_ERR_ARG, "proving key was loaded for a different shard");
    const uint64_t wb = local ? 0 : wlo, hb = local ? 0 : hlo;   // base-set index of this call's first point
    const bool overlapped = wcnt <= MAXC && hcnt <= MAXC && wcnt > 0 && hcnt > 0 && c->pinned;
    if (dist && world > 1 && !overlapped) return fail(c, SB_ERR_ARG, "distributed proving needs at least one point per rank and shards of at most 2^23 points");
    if (overlapped) {
        // Overlapped pipeline: the witness is sorted once (A, B1, B2 and C all multiply it, :84-97); the four bucket
        // pipelines run on their own streams so that the latency-bound tails (fold cascade, bucket reduction) of one
        // MSM hide under the throughput-bound accumulation of the next; the H scalars (QAP/NTT chain) are produced
        // concurrently on the main stream.  g_msm_tuning[2] != 0 serialises everything on one stream (profiling).
        const bool serial = g_msm_tuning[2] != 0;
        cudaStream_t s0 = c->stream;
        // schedule: main stream  : H2D, sort(witness), acc B2, acc A, acc B1, acc C, [join NTT chain], acc H
        //           aux[5] (hi)  : QAP -> iNTT -> coset NTT -> [exchange] -> joinABC -> sort(H scalars)
        //           aux[0..4](hi): the latency-bound tail of each MSM (fold, reduce, window sum, D2H)
        cudaStream_t sN = serial ? s0 : c->aux[5];
        MsmGeom gw = msm_geometry(wcnt, 32, c->fr_bits), gh = msm_geometry(hcnt, 32, c->fr_bits);
        const bool pre = k->tA != nullptr;
        if (pre) { gw = k->gpW; gw.first = wb; gh = k->gpH; gh.first = hb; }
        const size_t w1 = (size_t)gw.wsum_points() * G1.xyzz_bytes, w2 = (size_t)gw.wsum_points() * G2.xyzz_bytes, wh = (size_t)gh.wsum_points() * G1.xyzz_bytes;
        if (3 * w1 + w2 + wh + 64 > 256 * 1024 || 3 * w1 + w2 + wh > (size_t)8 * 80 * 4 * 96) return fail(c, SB_ERR_ARG, "window buffer too small");
        uint8_t* dws = (uint8_t*)k->dWsum; uint8_t* hws = c->pinned;
        uint64_t* hcounts = (uint64_t*)(c->pinned + 3 * w1 + w2 + wh);
        CU(c, cudaEventRecord(c->pev[0], s0));                       // witness resident
        if (sN != s0) CU(c, cudaStreamWaitEvent(sN, c->pev[0], 0));
        // NTT chain + sort of the H scalars on the side stream
        cudaStream_t saved = c->stream; c->stream = sN;
        rc = run_qap_ntt();
        MsmSorted sh;
        if (!rc) { rc = msm_sort_entries((const uint8_t*)tmp + hlo * 32, 32, hcnt, gh, c->sort_scratch2, sN, &sh, &c->stats); if (rc) rc = cuda_fail(c, (cudaError_t)rc, "msm_sort_entries"); }
        c->stream = saved;
        if (rc) return rc;
        CU(c, cudaEventRecord(c->pev[1], sN));
        // witness MSMs on the main stream
        MsmSorted sw;
        rc = msm_sort_entries((const uint8_t*)k->dW + wlo * 32, 32, wcnt, gw, c->sort_scratch, s0, &sw, &c->stats);
        if (rc) return cuda_fail(c, (cudaError_t)rc, "msm_sort_entries");
        tick(c, 2);
        struct Job { const GroupOps* G; const void* bases; size_t off; size_t len; uint8_t* dst; int tag; const MsmSorted* srt; const MsmGeom* g; };
        // order: A and B1 first (their results feed the host-side s*A + r*B1), then the long G2 MSM, C, and H last
        Job jobs[5] = {{&G1, pre ? k->tA : (const void*)((const uint8_t*)k->dA + wb * G1.aff_bytes), 0, w1, pA, SB_G1, &sw, &gw},
                       {&G1, pre ? k->tB1 : (const void*)((const uint8_t*)k->dB1 + wb * G1.aff_bytes), w1, w1, pB1, SB_G1, &sw, &gw},
                       {&G2, pre ? k->tB2 : (const void*)((const uint8_t*)k->dB2 + wb * G2.aff_bytes), 3 * w1, w2, pB2, SB_G2, &sw, &gw},
                       {&G1, pre ? k->tC : (const void*)((const uint8_t*)k->dC + wb * G1.aff_bytes), 2 * w1, w1, pC, SB_G1, &sw, &gw},
                       {&G1, pre ? k->tH : (const void*)((const uint8_t*)k->dH + hb * G1.aff_bytes), 3 * w1 + w2, wh, pH, SB_G1, &sh, &gh}};
        for (int i = 0; i < 5; i++) {
            cudaStream_t st = serial ? s0 : c->aux[i];
            if (i == 4 && sN != s0) CU(c, cudaStreamWaitEvent(s0, c->pev[1], 0));   // H needs the NTT chain
            c->stats.cur_tag = jobs[i].tag;
            rc = jobs[i].G->buckets(jobs[i].bases, *jobs[i].srt, c->bscr[i], s0, dws + jobs[i].off, &c->stats, st, c->pev[8 + i]);
            if (rc) return cuda_fail(c, (cudaError_t)rc, "msm_buckets");
            CU(c, cudaMemcpyAsync(hws + jobs[i].off, dws + jobs[i].off, jobs[i].len, cudaMemcpyDeviceToHost, st));
            if (i == 0) CU(c, cudaMemcpyAsync(&hcounts[0], sw.counts, 8, cudaMemcpyDeviceToHost, st));
            if (i == 4) CU(c, cudaMemcpyAsync(&hcounts[1], sh.counts, 8, cudaMemcpyDeviceToHost, st));
            CU(c, cudaEventRecord(c->pev[2 + i], st));
        }
        tick(c, 3);
        // host recombination as each MSM lands (overlaps with the MSMs still running)
        for (int i = 0; i < 5; i++) {
            CU(c, cudaEventSynchronize(c->pev[2 + i]));
            jobs[i].G->combine(hws + jobs[i].off, *jobs[i].g, jobs[i].dst);
            if (ps && i == 0) G1.times(pA, ps->sp, 32, sA.data());      // s * A   (src/groth16_prove.js:117: pi_c += s*pi_a)
            if (ps && i == 1) G1.times(pB1, ps->rp, 32, rB1.data());    // r * B1  (:118)
        }
        // join the side streams back into the main stream
        if (!serial) { for (int i = 0; i < 5; i++) CU(c, cudaStreamWaitEvent(s0, c->pev[2 + i], 0)); CU(c, cudaStreamWaitEvent(s0, c->pev[1], 0)); }
        c->stat[4] += 3.0 * (double)hcounts[0] + (double)hcounts[1]; c->stat[5] += (double)hcounts[0];
    } else {
    rc = run_qap_ntt(); if (rc) return rc;
    tick(c, 2);
    for (uint64_t off = 0; off < wcnt; off += MAXC) {
        uint64_t cn = std::min(MAXC, wcnt - off), base = wb + off;
        MsmGeom g = msm_geometry(cn, 32, c->fr_bits);
        MsmSorted s;
        rc = msm_sort_entries((const uint8_t*)k->dW + (wlo + off) * 32, 32, cn, g, c->sort_scratch, c->stream, &s, &c->stats);
        if (rc) return cuda_fail(c, (cudaError_t)rc, "msm_sort_entries");
        uint8_t* ws = (uint8_t*)k->dWsum;
        size_t w1 = (size_t)g.wsum_points() * G1.xyzz_bytes, w2 = (size_t)g.wsum_points() * G2.xyzz_bytes;
        if (3 * w1 + w2 > (size_t)8 * 80 * 4 * 96) return fail(c, SB_ERR_ARG, "window buffer too small");
        c->stats.cur_tag = SB_G1;
        rc = G1.buckets((const uint8_t*)k->dA + base * G1.aff_bytes, s, c->bucket_scratch, c->stream, ws, &c->stats, nullptr, nullptr); if (rc) return cuda_fail(c, (cudaError_t)rc, "msm A");
        rc = G1.buckets((const uint8_t*)k->dB1 + base * G1.aff_bytes, s, c->bucket_scratch, c->stream, ws + w1, &c->stats, nullptr, nullptr); if (rc) return cuda_fail(c, (cudaError_t)rc, "msm B1");
        rc = G1.buckets((const uint8_t*)k->dC + base * G1.aff_bytes, s, c->bucket_scratch, c->stream, ws + 2 * w1, &c->stats, nullptr, nullptr); if (rc) return cuda_fail(c, (cudaError_t)rc, "msm C");
        c->stats.cur_tag = SB_G2;
        rc = G2.buckets((const uint8_t*)k->dB2 + base * G2.aff_bytes, s, c->bucket_scratch, c->stream, ws + 3 * w1, &c->stats, nullptr, nullptr); if (rc) return cuda_fail(c, (cudaError_t)rc, "msm B2");
        std::vector<uint8_t> hw(3 * w1 + w2);
        uint64_t entries = 0;
        CU(c, cudaMemcpyAsync(hw.data(), ws, hw.size(), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(&entries, s.counts, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        c->stat[4] += 3.0 * (double)entries; c->stat[5] += (double)entries;
        G1.combine(hw.data(), g, pA); G1.combine(hw.data() + w1, g, pB1); G1.combine(hw.data() + 2 * w1, g, pC); G2.combine(hw.data() + 3 * w1, g, pB2);
    }
    tick(c, 3);
    if (hcnt) {
        rc = msm_dev_accumulate(c, G1, (const uint8_t*)k->dH + hb * G1.aff_bytes, (const uint8_t*)tmp + hlo * 32, 32, hcnt, pH);
        if (rc) return rc;
    }
    if (ps) { G1.times(pA, ps->sp, 32, sA.data()); G1.times(pB1, ps->rp, 32, rB1.data()); }
    }
    if (ps) {   // C' = C + H + s*A + r*B1;  the B1 and H slots are spent
        G1.add(pC, pH); G1.add(pC, sA.data()); G1.add(pC, rB1.data());
        memset(pB1, 0, G1.xyzz_bytes); memset(pH, 0, G1.xyzz_bytes);
    }
    tick(c, 4);
    cudaEventSynchronize(c->ev[4]);
    prof_end(c);
    c->last_ms[0] = elapsed(c, 0, 4); c->last_ms[1] = elapsed(c, 0, 1); c->last_ms[2] = elapsed(c, 1, 2); c->last_ms[3] = elapsed(c, 2, 3); c->last_ms[4] = elapsed(c, 3, 4);
    return 0;
}

// host part: proof assembly, src/groth16_prove.js:103-132

struct VkPoints { const uint8_t *alpha1, *beta1, *beta2, *delta1, *delta2; };
static void plain_scalars(int curve, const uint8_t r[32], const uint8_t s[32], uint8_t rp[32], uint8_t sp[32], uint8_t rsp[32], bool negate_rs) {
    uint8_t rs[32];
    if (curve == SB_BN254) {
        fr_from_mont_bytes<BnFr>(r, rp); fr_from_mont_bytes<BnFr>(s, sp);
        Fp<BnFr> a, b; memcpy(&a, r, 32); memcpy(&b, s, 32); a = Fp<BnFr>::mul(a, b); if (negate_rs) a = Fp<BnFr>::neg(a); memcpy(rs, &a, 32);
        fr_from_mont_bytes<BnFr>(rs, rsp);
    } else {
        fr_from_mont_bytes<BlsFr>(r, rp); fr_from_mont_bytes<BlsFr>(s, sp);
        Fp<BlsFr> a, b; memcpy(&a, r, 32); memcpy(&b, s, 32); a = Fp<BlsFr>::mul(a, b); if (negate_rs) a = Fp<BlsFr>::neg(a); memcpy(rs, &a, 32);
        fr_from_mont_bytes<BlsFr>(rs, rsp);
    }
}
static int groth16_assemble_host(int curve, const GroupOps& G1, const GroupOps& G2, const VkPoints& vk, const uint8_t* partials,
                                 const uint8_t r[32], const uint8_t s[32], uint8_t* proof);
static int groth16_assemble(sb_ctx* c, Groth16Key* k, const uint8_t* partials, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) {
    VkPoints vk{k->alpha1.data(), k->beta1.data(), k->beta2.data(), k->delta1.data(), k->delta2.data()};
    return groth16_assemble_host(c->curve, c->g1, c->g2, vk, partials, r, s, proof);
}
static int groth16_assemble_host(int curve, const GroupOps& G1, const GroupOps& G2, const VkPoints& vk, const uint8_t* partials,
                                 const uint8_t r[32], const uint8_t s[32], uint8_t* proof) {
    const uint32_t x1 = G1.xyzz_bytes, x2 = G2.xyzz_bytes;
    std::vector<uint8_t> A(partials, partials + x1), B1(partials + x1, partials + 2 * x1), C(partials + 2 * x1, partials + 3 * x1),
        H(partials + 3 * x1, partials + 4 * x1), B2(partials + 4 * x1, partials + 4 * x1 + x2);
    uint8_t rp[32], sp[32], rsp[32];
    plain_scalars(curve, r, s, rp, sp, rsp, true);
    std::vector<uint8_t> t1(x1), t2(x2), d1(x1), d2(x2), pt(x1), pt2(x2);
    G1.from_affine(vk.delta1, d1.data()); G2.from_affine(vk.delta2, d2.data());
    // pi_a = A + alpha1 + r*delta1
    G1.from_affine(vk.alpha1, pt.data()); G1.add(A.data(), pt.data());
    G1.times(d1.data(), rp, 32, t1.data()); G1.add(A.data(), t1.data());
    // pi_b = B2 + beta2 + s*delta2
    G2.from_affine(vk.beta2, pt2.data()); G2.add(B2.data(), pt2.data());
    G2.times(d2.data(), sp, 32, t2.data()); G2.add(B2.data(), t2.data());
    // pib1 = B1 + beta1 + s*delta1
    G1.from_affine(vk.beta1, pt.data()); G1.add(B1.data(), pt.data());
    G1.times(d1.data(), sp, 32, t1.data()); G1.add(B1.data(), t1.data());
    // pi_c = C + H + s*pi_a + r*pib1 - rs*delta1
    G1.add(C.data(), H.data());
    G1.times(A.data(), sp, 32, t1.data()); G1.add(C.data(), t1.data());
    G1.times(B1.data(), rp, 32, t1.data()); G1.add(C.data(), t1.data());
    G1.times(d1.data(), rsp, 32, t1.data()); G1.add(C.data(), t1.data());
    G1.to_affine(A.data(), proof);
    G2.to_affine(B2.data(), proof + G1.aff_bytes);
    G1.to_affine(C.data(), proof + G1.aff_bytes + G2.aff_bytes);
    return 0;
}

// The same assembly split so that nothing but three additions and three normalisations follows the last MSM:
//   pi_a = A + [alpha1 + r*delta1],  pi_b = B2 + [beta2 + s*delta2],
//   pi_c = C + H + s*pi_a + r*pib1 - rs*delta1 = [C + H + s*A + r*B1] + [s*alpha1 + r*beta1 + rs*delta1]
// The bracketed fixed parts depend only on the key and (r, s): a helper thread computes them while the GPU works;
// the C bracket is folded by groth16_device (ProofScalars) as A and B1 land.  Same group elements, same proof bytes.
struct FixedParts { std::vector<uint8_t> Fa, Fb, Fc; };
static FixedParts groth16_fixed_parts(int curve, const GroupOps& G1, const GroupOps& G2, const VkPoints vk, const uint8_t* r, const uint8_t* s) {
    const uint32_t x1 = G1.xyzz_bytes, x2 = G2.xyzz_bytes;
    uint8_t rp[32], sp[32], rsp[32];
    plain_scalars(curve, r, s, rp, sp, rsp, false);
    FixedParts f; f.Fa.assign(x1, 0); f.Fb.assign(x2, 0); f.Fc.assign(x1, 0);
    std::vector<uint8_t> a1(x1), b1(x1), d1(x1), b2(x2), d2(x2), t1(x1), t2(x2);
    G1.from_affine(vk.alpha1, a1.data()); G1.from_affine(vk.beta1, b1.data()); G1.from_affine(vk.delta1, d1.data());
    G2.from_affine(vk.beta2, b2.data()); G2.from_affine(vk.delta2, d2.data());
    std::future<void> g2 = std::async(std::launch::async, [&]() { G2.times(d2.data(), sp, 32, t2.data()); });   // the one G2 multiple, on its own thread
    G1.times(d1.data(), rp, 32, t1.data()); f.Fa = a1; G1.add(f.Fa.data(), t1.data());
    G1.times(a1.data(), sp, 32, f.Fc.data());
    G1.times(b1.data(), rp, 32, t1.data()); G1.add(f.Fc.data(), t1.data());
    G1.times(d1.data(), rsp, 32, t1.data()); G1.add(f.Fc.data(), t1.data());
    g2.get();
    f.Fb = b2; G2.add(f.Fb.data(), t2.data());
    return f;
}
static void groth16_finish_folded(const GroupOps& G1, const GroupOps& G2, const FixedParts& f, const uint8_t* partials, uint8_t* proof) {
    const uint32_t x1 = G1.xyzz_bytes, x2 = G2.xyzz_bytes;
    std::vector<uint8_t> A(partials, partials + x1), C(partials + 2 * x1, partials + 3 * x1), B2(partials + 4 * x1, partials + 4 * x1 + x2);
    G1.add(A.data(), f.Fa.data()); G2.add(B2.data(), f.Fb.data()); G1.add(C.data(), f.Fc.data());
    G1.to_affine(A.data(), proof);
    G2.to_affine(B2.data(), proof + G1.aff_bytes);
    G1.to_affine(C.data(), proof + G1.aff_bytes + G2.aff_bytes);
}
static int groth16_prove_folded(sb_ctx* c, Groth16Key* k, const uint8_t* witness, uint64_t n_witness, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) {
    VkPoints vk{k->alpha1.data(), k->beta1.data(), k->beta2.data(), k->delta1.data(), k->delta2.data()};
    const int curve = c->curve; const GroupOps G1 = c->g1, G2 = c->g2;
    std::future<FixedParts> fixed = std::async(std::launch::async, [=]() { return groth16_fixed_parts(curve, G1, G2, vk, r, s); });
    ProofScalars ps; uint8_t rsp[32]; plain_scalars(curve, r, s, ps.rp, ps.sp, rsp, false);
    std::vector<uint8_t> partials(sb_groth16_partials_bytes(c));
    int rc = groth16_device(c, k, witness, n_witness, 0, 1, partials.data(), &ps, false);
    FixedParts f = fixed.get();
    if (rc) return rc;
    groth16_finish_folded(c->g1, c->g2, f, partials.data(), proof);
    return 0;
}

int sb_groth16_prove(sb_ctx* c, uint64_t h, const uint8_t* witness, uint64_t n_witness, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    if (k->n_shards > 1) return fail(c, SB_ERR_ARG, "proving key was loaded sharded: use sb_groth16_prove_shard + sb_groth16_finish");
    if (!witness || !r || !s || !proof) return fail(c, SB_ERR_ARG, "null argument");
    return groth16_prove_folded(c, k, witness, n_witness, r, s, proof);
}
int sb_groth16_prove_resident(sb_ctx* c, uint64_t h, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    if (k->n_shards > 1) return fail(c, SB_ERR_ARG, "proving key was loaded sharded: use sb_groth16_prove_shard + sb_groth16_finish");
    if (!r || !s || !proof) return fail(c, SB_ERR_ARG, "null argument");
    return groth16_prove_folded(c, k, nullptr, k->nVars, r, s, proof);
}
int sb_groth16_prove_shard(sb_ctx* c, uint64_t h, const uint8_t* witness, uint64_t n_witness, int shard, int n_shards, uint8_t* partials_out) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(c, SB_ERR_ARG, "invalid shard");
    return groth16_device(c, k, witness, n_witness, shard, n_shards, partials_out);
}
int sb_groth16_finish(sb_ctx* c, uint64_t h, const uint8_t* all, int n_shards, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    const GroupOps& G1 = c->g1; const GroupOps& G2 = c->g2;
    const uint32_t x1 = G1.xyzz_bytes, pb = sb_groth16_partials_bytes(c);
    std::vector<uint8_t> acc(pb, 0);
    for (int i = 0; i < n_shards; i++) {
        const uint8_t* p = all + (size_t)i * pb;
        for (int j = 0; j < 4; j++) G1.add(acc.data() + j * x1, p + j * x1);
        G2.add(acc.data() + 4 * x1, p + 4 * x1);
    }
    return groth16_assemble(c, k, acc.data(), r, s, proof);
}

// One proof across the ranks of a communicator (collective: every rank calls it with the same witness, r and s).
// witness may be null on every rank to reuse the resident one.  proof_affine_out may be null on ranks that do not need
// the proof; ranks that pass a buffer all receive the same bytes.
int sb_groth16_prove_dist(sb_ctx* c, uint64_t h, const uint8_t* witness, uint64_t n_witness, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    if (!c->comm) return fail(c, SB_ERR_ARG, "context has no communicator: call sb_comm_init_rank first");
    if (!r || !s) return fail(c, SB_ERR_ARG, "null argument");
    NcclApi* nc = nccl_api(nullptr);
    VkPoints vk{k->alpha1.data(), k->beta1.data(), k->beta2.data(), k->delta1.data(), k->delta2.data()};
    const int curve = c->curve; const GroupOps G1 = c->g1, G2 = c->g2;
    std::future<FixedParts> fixed;
    if (proof) fixed = std::async(std::launch::async, [=]() { return groth16_fixed_parts(curve, G1, G2, vk, r, s); });
    ProofScalars ps; uint8_t rsp[32]; plain_scalars(curve, r, s, ps.rp, ps.sp, rsp, false);
    const size_t pb = sb_groth16_partials_bytes(c);
    uint8_t* mine = c->h_xchg + pb * c->world;
    int rc = groth16_device(c, k, witness, n_witness, c->rank, c->world, mine, &ps, true);
    if (rc) { if (proof) fixed.get(); return rc; }
    cudaError_t e = cudaMemcpyAsync((uint8_t*)c->d_xchg + pb * c->rank, mine, pb, cudaMemcpyHostToDevice, c->stream);
    ncclResult_t nr = ncclSuccess;
    if (e == cudaSuccess) nr = nc->AllGather((const uint8_t*)c->d_xchg + pb * c->rank, c->d_xchg, pb, ncclUint8, c->comm, c->stream);
    if (e == cudaSuccess && nr == ncclSuccess && proof) e = cudaMemcpyAsync(c->h_xchg, c->d_xchg, pb * c->world, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (proof) {
        FixedParts f = fixed.get();
        if (e == cudaSuccess && nr == ncclSuccess) {
            const uint32_t x1 = G1.xyzz_bytes;
            std::vector<uint8_t> acc(pb, 0);
            for (int i = 0; i < c->world; i++) {
                const uint8_t* p = c->h_xchg + (size_t)i * pb;
                G1.add(acc.data(), p); G1.add(acc.data() + 2 * x1, p + 2 * x1); G2.add(acc.data() + 4 * x1, p + 4 * x1);
            }
            groth16_finish_folded(G1, G2, f, acc.data(), proof);
        }
    }
    if (nr != ncclSuccess) return fail(c, SB_ERR_CUDA, std::string("ncclAllGather: ") + nc->GetErrorString(nr));
    if (e != cudaSuccess) return cuda_fail(c, e, "partial exchange");
    return 0;
}

// ---- single-process multi-GPU convenience (what a Node addon calls): one context per device, one host thread per
// context inside each call.  SURVEY §8b: sb_create(curve, device_ids, n_devices) with the communicator built here.
int sb_create_multi(int curve, const int* device_ids, int n_devices, sb_ctx** out) {
    if (!device_ids || !out || n_devices < 1 || n_devices > 64) return SB_ERR_ARG;
    for (int i = 0; i < n_devices; i++) out[i] = nullptr;
    int rc = 0;
    for (int i = 0; i < n_devices && !rc; i++) rc = sb_create(curve, device_ids[i], &out[i]);
    uint8_t id[128];
    if (!rc && n_devices > 1) rc = sb_comm_unique_id(id);
    if (!rc && n_devices > 1) {
        std::vector<std::future<int>> f;
        for (int i = 0; i < n_devices; i++) f.push_back(std::async(std::launch::async, [=]() { return sb_comm_init_rank(out[i], n_devices, i, id); }));
        for (auto& x : f) { int r = x.get(); if (r && !rc) rc = r; }
    }
    if (rc) { for (int i = 0; i < n_devices; i++) { if (out[i]) sb_destroy(out[i]); out[i] = nullptr; } }
    return rc;
}
int sb_groth16_load_multi(sb_ctx* const* ctxs, int n, const uint8_t* zkey, uint64_t zkey_len, uint64_t* handles) {
    if (!ctxs || !zkey || !handles || n < 1) return SB_ERR_ARG;
    std::vector<std::future<int>> f;
    for (int i = 0; i < n; i++) f.push_back(std::async(std::launch::async, [=]() { return sb_groth16_load_sharded(ctxs[i], zkey, zkey_len, i, n, &handles[i]); }));
    int rc = 0; for (auto& x : f) { int r = x.get(); if (r && !rc) rc = r; }
    return rc;
}
int sb_groth16_prove_multi(sb_ctx* const* ctxs, const uint64_t* handles, int n, const uint8_t* witness, uint64_t n_witness,
                           const uint8_t r[32], const uint8_t s[32], uint8_t* proof_affine_out) {
    if (!ctxs || !handles || n < 1 || !proof_affine_out) return SB_ERR_ARG;
    if (n == 1) return sb_groth16_prove(ctxs[0], handles[0], witness, n_witness, r, s, proof_affine_out);
    std::vector<std::future<int>> f;
    for (int i = 0; i < n; i++)
        f.push_back(std::async(std::launch::async, [=]() { return sb_groth16_prove_dist(ctxs[i], handles[i], witness, n_witness, r, s, i == 0 ? proof_affine_out : nullptr); }));
    int rc = 0; for (auto& x : f) { int r2 = x.get(); if (r2 && !rc) rc = r2; }
    return rc;
}

// ---- host-only helpers (no context, no device): the combine/assembly half of the multi-GPU path, testable on CPU
static void host_ops(int curve, GroupOps& g1, GroupOps& g2) {
    if (curve == SB_BN254) { g1 = SB_GROUP_OPS(bn254_g1, 64); g2 = SB_GROUP_OPS(bn254_g2, 128); }
    else { g1 = SB_GROUP_OPS(bls12381_g1, 96); g2 = SB_GROUP_OPS(bls12381_g2, 192); }
}
int sb_host_sum_partials(int curve, int group, const uint8_t* partials, int count, uint8_t* out_jacobian) {
    if ((curve != SB_BN254 && curve != SB_BLS12_381) || (group != SB_G1 && group != SB_G2) || count < 0) return SB_ERR_ARG;
    GroupOps g1, g2; host_ops(curve, g1, g2);
    const GroupOps& G = group == SB_G1 ? g1 : g2;
    std::vector<uint8_t> acc(G.xyzz_bytes, 0);
    for (int i = 0; i < count; i++) G.add(acc.data(), partials + (size_t)i * G.xyzz_bytes);
    G.to_jacobian(acc.data(), out_jacobian);
    return 0;
}
int sb_host_partial_from_affine(int curve, int group, const uint8_t* affine, uint8_t* partial_out) {
    if ((curve != SB_BN254 && curve != SB_BLS12_381) || (group != SB_G1 && group != SB_G2)) return SB_ERR_ARG;
    GroupOps g1, g2; host_ops(curve, g1, g2);
    (group == SB_G1 ? g1 : g2).from_affine(affine, partial_out);
    return 0;
}
uint32_t sb_host_partial_bytes(int curve, int group) {
    GroupOps g1, g2; if (curve != SB_BN254 && curve != SB_BLS12_381) return 0; host_ops(curve, g1, g2);
    return group == SB_G1 ? g1.xyzz_bytes : g2.xyzz_bytes;
}
int sb_host_groth16_finish(int curve, const uint8_t* vk_alpha1, const uint8_t* vk_beta1, const uint8_t* vk_beta2,
                           const uint8_t* vk_delta1, const uint8_t* vk_delta2, const uint8_t* partials_all_ranks, int n_shards,
                           const uint8_t r[32], const uint8_t s[32], uint8_t* proof_affine_out) {
    if ((curve != SB_BN254 && curve != SB_BLS12_381) || n_shards < 1) return SB_ERR_ARG;
    GroupOps G1, G2; host_ops(curve, G1, G2);
    const uint32_t x1 = G1.xyzz_bytes, pb = 4 * G1.xyzz_bytes + G2.xyzz_bytes;
    std::vector<uint8_t> acc(pb, 0);
    for (int i = 0; i < n_shards; i++) {
        const uint8_t* p = partials_all_ranks + (size_t)i * pb;
        for (int j = 0; j < 4; j++) G1.add(acc.data() + j * x1, p + j * x1);
        G2.add(acc.data() + 4 * x1, p + 4 * x1);
    }
    VkPoints vk{vk_alpha1, vk_beta1, vk_beta2, vk_delta1, vk_delta2};
    return groth16_assemble_host(curve, G1, G2, vk, acc.data(), r, s, proof_affine_out);
}
// point range of shard `shard` of `n_shards` over `total` points (the split sb_groth16_prove_shard uses)
void sb_shard_range(uint64_t total, int shard, int n_shards, uint64_t* first, uint64_t* count) {
    uint64_t per = (total + n_shards - 1) / n_shards, lo = std::min(total, per * (uint64_t)shard);
    *first = lo; *count = std::min(total - lo, per);
}

int sb_groth16_prove_wtns(sb_ctx* c, uint64_t h, const uint8_t* w, uint64_t wlen, const uint8_t r[32], const uint8_t s[32], uint8_t* proof) { SB_LOCK(c);
    Groth16Key* k = get_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid groth16 handle");
    std::map<uint32_t, Section> secs;
    int rc = parse_binfile(c, w, wlen, "wtns", 2, secs); if (rc) return rc;
    if (!secs[1].present || !secs[2].present) return fail(c, SB_ERR_FORMAT, "Missing section");
    const uint8_t* hd = w + secs[1].pos;
    if (secs[1].len < 4) return fail(c, SB_ERR_FORMAT, "wtns header too short");
    uint32_t n8; memcpy(&n8, hd, 4);
    if (secs[1].len < 8 + (uint64_t)n8) return fail(c, SB_ERR_FORMAT, "wtns header too short");
    if (!modulus_matches(hd + 4, n8, c->curve, true)) return fail(c, SB_ERR_ARG, "Curve of the witness does not match the curve of the proving key");
    uint32_t nw; memcpy(&nw, hd + 4 + n8, 4);
    if (secs[2].len != (uint64_t)nw * n8) return fail(c, SB_ERR_FORMAT, "Invalid witness section size");
    return sb_groth16_prove(c, h, w + secs[2].pos, nw, r, s, proof);
}

}  // extern "C"

// ================================================================================================================
// PLONK (src/plonk_prove.js) — templates live outside the extern "C" block
#include "api_plonk.inl"
#include "api_fflonk.inl"

extern "C" {

int sb_plonk_load(sb_ctx* c, const uint8_t* zkey, uint64_t len, uint64_t* handle) { SB_LOCK(c);
    if (!c || !zkey || !handle) return SB_ERR_ARG;
    cudaSetDevice(c->device);
    return c->curve == SB_BN254 ? plonk_load_impl<BnFr>(c, zkey, len, handle) : plonk_load_impl<BlsFr>(c, zkey, len, handle);
}
// maps the file read-only and hands it to the byte loader: the sections are read once, front to back, through the pinned
// staging buffers (h2d), so the key never sits in anonymous host memory
static int load_mapped(sb_ctx* c, const char* path, uint64_t* handle, int (*load)(sb_ctx*, const uint8_t*, uint64_t, uint64_t*)) {
    if (!c || !path || !handle) return SB_ERR_ARG;
    int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(c, SB_ERR_FORMAT, std::string("cannot open ") + path);
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); return fail(c, SB_ERR_FORMAT, std::string("cannot stat ") + path); }
    void* p = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (p == MAP_FAILED) return fail(c, SB_ERR_FORMAT, std::string("cannot map ") + path);
    madvise(p, (size_t)st.st_size, MADV_SEQUENTIAL);
    int rc = load(c, (const uint8_t*)p, (uint64_t)st.st_size, handle);
    munmap(p, (size_t)st.st_size);
    return rc;
}
int sb_plonk_load_file(sb_ctx* c, const char* path, uint64_t* handle) { SB_LOCK(c); return load_mapped(c, path, handle, sb_plonk_load); }
static PlonkKeyDev* get_plonk_key(sb_ctx* c, uint64_t h) { return (c && h >= 1 && h <= c->plonk_keys.size()) ? c->plonk_keys[h - 1] : nullptr; }
int sb_plonk_info(sb_ctx* c, uint64_t h, uint32_t* n_vars, uint32_t* n_public, uint32_t* domain_size, uint32_t* n_additions) { SB_LOCK(c);
    PlonkKeyDev* k = get_plonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid plonk handle");
    if (n_vars) *n_vars = k->z.nVars; if (n_public) *n_public = k->z.nPublic; if (domain_size) *domain_size = k->z.n; if (n_additions) *n_additions = k->z.nAdditions;
    return 0;
}
uint32_t sb_plonk_proof_bytes(sb_ctx* c) { return c ? 9 * c->g1.aff_bytes + 6 * 32 : 0; }
int sb_plonk_prove(sb_ctx* c, uint64_t h, const uint8_t* witness, uint64_t n_witness, const uint8_t* blinders, uint8_t* proof) { SB_LOCK(c);
    PlonkKeyDev* k = get_plonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid plonk handle");
    if (!witness || !blinders || !proof) return fail(c, SB_ERR_ARG, "null argument");
    cudaSetDevice(c->device);
    return c->curve == SB_BN254 ? plonk_prove_impl<BnFq, BnFr>(c, k, witness, n_witness, blinders, proof)
                                : plonk_prove_impl<BlsFq, BlsFr>(c, k, witness, n_witness, blinders, proof);
}
int sb_plonk_prove_resident(sb_ctx* c, uint64_t h, const uint8_t* blinders, uint8_t* proof) { SB_LOCK(c);
    PlonkKeyDev* k = get_plonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid plonk handle");
    if (!blinders || !proof) return fail(c, SB_ERR_ARG, "null argument");
    if (!k->n_wit_resident) return fail(c, SB_ERR_ARG, "no witness resident for this proving key: call sb_plonk_prove first");
    cudaSetDevice(c->device);
    return c->curve == SB_BN254 ? plonk_prove_impl<BnFq, BnFr>(c, k, nullptr, 0, blinders, proof)
                                : plonk_prove_impl<BlsFq, BlsFr>(c, k, nullptr, 0, blinders, proof);
}
int sb_plonk_release(sb_ctx* c, uint64_t h) { SB_LOCK(c);
    PlonkKeyDev* k = get_plonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid plonk handle");
    cudaSetDevice(c->device); cudaStreamSynchronize(c->stream);
    plonk_free_key(k); c->plonk_keys[h - 1] = nullptr;
    return 0;
}

// ---- fflonk (src/fflonk_prove.js)
int sb_fflonk_load(sb_ctx* c, const uint8_t* zkey, uint64_t len, uint64_t* handle) { SB_LOCK(c);
    if (!c || !zkey || !handle) return SB_ERR_ARG;
    if (c->curve != SB_BN254) return fail(c, SB_ERR_ARG, "fflonk is defined on bn128 only (src/fflonk_setup.js:534-557)");
    cudaSetDevice(c->device);
    return fflonk_load_impl<BnFr>(c, zkey, len, handle);
}
int sb_fflonk_load_file(sb_ctx* c, const char* path, uint64_t* handle) { SB_LOCK(c); return load_mapped(c, path, handle, sb_fflonk_load); }
static FflonkKeyDev* get_fflonk_key(sb_ctx* c, uint64_t h) { return (c && h >= 1 && h <= c->fflonk_keys.size()) ? c->fflonk_keys[h - 1] : nullptr; }
int sb_fflonk_info(sb_ctx* c, uint64_t h, uint32_t* n_vars, uint32_t* n_public, uint32_t* domain_size, uint32_t* n_additions) { SB_LOCK(c);
    FflonkKeyDev* k = get_fflonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid fflonk handle");
    if (n_vars) *n_vars = k->z.nVars; if (n_public) *n_public = k->z.nPublic; if (domain_size) *domain_size = k->z.n; if (n_additions) *n_additions = k->z.nAdditions;
    return 0;
}
uint32_t sb_fflonk_proof_bytes(sb_ctx* c) { return c ? 4 * c->g1.aff_bytes + 16 * 32 : 0; }
int sb_fflonk_prove(sb_ctx* c, uint64_t h, const uint8_t* witness, uint64_t n_witness, const uint8_t* blinders, uint8_t* proof) { SB_LOCK(c);
    FflonkKeyDev* k = get_fflonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid fflonk handle");
    if (!witness || !blinders || !proof) return fail(c, SB_ERR_ARG, "null argument");
    cudaSetDevice(c->device);
    return fflonk_prove_impl<BnFq, BnFr>(c, k, witness, n_witness, blinders, proof);
}
int sb_fflonk_prove_resident(sb_ctx* c, uint64_t h, const uint8_t* blinders, uint8_t* proof) { SB_LOCK(c);
    FflonkKeyDev* k = get_fflonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid fflonk handle");
    if (!blinders || !proof) return fail(c, SB_ERR_ARG, "null argument");
    if (!k->n_wit_resident) return fail(c, SB_ERR_ARG, "no witness resident for this proving key: call sb_fflonk_prove first");
    cudaSetDevice(c->device);
    return fflonk_prove_impl<BnFq, BnFr>(c, k, nullptr, 0, blinders, proof);
}
int sb_fflonk_release(sb_ctx* c, uint64_t h) { SB_LOCK(c);
    FflonkKeyDev* k = get_fflonk_key(c, h); if (!k) return fail(c, SB_ERR_ARG, "invalid fflonk handle");
    cudaSetDevice(c->device); cudaStreamSynchronize(c->stream);
    fflonk_free_key(k); c->fflonk_keys[h - 1] = nullptr;
    return 0;
}

}  // extern "C"
