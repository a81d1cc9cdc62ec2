// CPU model of the batched-affine rounds of msm_pair.cuh: the slot layout of k_pair_prefix / k_pair_apply (slot
// j = k*T + t of thread t, prefix products in slot order, back-substitution from the last slot), the output positions by
// an exclusive sum of the per-slot counts, and the pair arithmetic itself through the very templates the kernels run
// (pair_kind, pair_sum on fp.cuh / ec.cuh).  The shared inversion is a plain field inversion per thread product here.
// Sorted lists of real curve points (multiples of the generator) with odd runs, runs across thread boundaries, points at
// infinity, P + P (also across rounds) and P + (-P) go through several rounds; after every round the list must still be
// sorted, and every bucket sum (XYZZ mixed additions, pinned to the oracle by host_fp_check.cpp) must be unchanged.
// Built and run by tests/test_host_templates.py:  g++ -O2 -std=c++17
#include <cstdio>
#include <cstring>
#include <vector>
#include "../../snarkjs_b200/csrc/ec.cuh"
#include "../../snarkjs_b200/csrc/msm_pair.cuh"
using namespace sb;

static uint64_t rng_state = 0x2545F4914F6CDD1Dull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

template <class P> static Fp<P> from_hex(const char* hex) {
    Fp<P> a = Fp<P>::zero();
    const int len = (int)strlen(hex);
    for (int i = 0; i < len; i++) {
        const char ch = hex[len - 1 - i];
        const uint32_t d = (ch >= '0' && ch <= '9') ? ch - '0' : ch - 'a' + 10;
        a.v[i / 8] |= d << (4 * (i % 8));
    }
    return Fp<P>::to_mont(a);
}
template <class F> static F finv(const F& a) { return F::inv(a); }

template <class F> static Affine<F> to_affine(const XYZZ<F>& p) {
    Affine<F> a;
    if (p.is_inf()) { a.x = F::zero(); a.y = F::zero(); return a; }
    a.x = F::mul(p.x, finv(p.zz)); a.y = F::mul(p.y, finv(p.zzz));
    return a;
}
template <class F> static Affine<F> mul_small(const Affine<F>& g, uint32_t k) {
    XYZZ<F> r = XYZZ<F>::inf();
    for (int b = 31; b >= 0; b--) { r = XYZZ<F>::dbl(r); if ((k >> b) & 1) r.add_affine(g.x, g.y, F::one()); }
    return to_affine(r);
}
template <class T> static bool same(const T& a, const T& b) { return memcmp(&a, &b, sizeof(T)) == 0; }
static int g_bad_inverse = 0;

// bucket sums of a sorted list, as affine points (buckets absent from the list are the point at infinity)
template <class F> static std::vector<Affine<F>> bucket_sums(const std::vector<uint32_t>& keys, const std::vector<Affine<F>>& pts, uint32_t NB) {
    std::vector<XYZZ<F>> acc(NB, XYZZ<F>::inf());
    for (size_t i = 0; i < keys.size(); i++)
        if (!pts[i].is_inf()) acc[keys[i]].add_affine(pts[i].x, pts[i].y, F::one());
    std::vector<Affine<F>> out(NB);
    for (uint32_t b = 0; b < NB; b++) out[b] = to_affine(acc[b]);
    return out;
}

// one round with T threads of K slots (K * T >= ceil(n/2)), mirroring k_pair_prefix / scan / k_pair_apply
template <class F> static void round_model(std::vector<uint32_t>& keys, std::vector<Affine<F>>& pts, uint64_t T, uint32_t K, int& nadd, int& ndbl) {
    const uint64_t n = keys.size(), J = (n + 1) / 2;
    std::vector<F> pre(J), tprod(T), invp(T);
    std::vector<uint32_t> outc(J + 1, 0), pos(J + 1, 0);
    for (uint64_t t = 0; t < T; t++) {                                     // k_pair_prefix
        F acc = F::one();
        for (uint32_t k = 0; k < K; k++) {
            const uint64_t j = k * T + t;
            if (j >= J) break;
            const uint64_t s = 2 * j;
            outc[j] = 1;
            if (s + 1 < n) {
                if (keys[s] != keys[s + 1]) outc[j] = 2;
                else {
                    F den; const int kind = pair_kind<F>(pts[s].x, pts[s].y, pts[s + 1].x, pts[s + 1].y, den);
                    if (kind == PAIR_ADD || kind == PAIR_DBL) { pre[j] = acc; acc = F::mul(acc, den); }
                }
            }
        }
        tprod[t] = acc;
    }
    for (uint64_t j = 0; j < J; j++) pos[j + 1] = pos[j] + outc[j];      // cub exclusive sum; pos[J] = new length
    for (uint64_t t = 0; t < T; t++) invp[t] = finv(tprod[t]);            // k_pair_invert
    std::vector<uint32_t> nk(pos[J]); std::vector<Affine<F>> np(pos[J]);
    for (uint64_t t = 0; t < T; t++) {                                     // k_pair_apply
        F running = invp[t];
        for (int k = (int)K - 1; k >= 0; k--) {
            const uint64_t j = (uint64_t)k * T + t;
            if (j >= J) continue;
            const uint64_t s = 2 * j; const uint32_t o = pos[j];
            Affine<F> a = pts[s];
            if (s + 1 < n) {
                const Affine<F> b = pts[s + 1];
                if (keys[s + 1] != keys[s]) { np[o + 1] = b; nk[o + 1] = keys[s + 1]; }
                else {
                    F den; const int kind = pair_kind<F>(a.x, a.y, b.x, b.y, den);
                    F inv = den;
                    if (kind == PAIR_ADD || kind == PAIR_DBL) {
                        inv = F::mul(running, pre[j]); running = F::mul(running, den);
                        if (!same(F::mul(inv, den), F::one())) { g_bad_inverse++; printf("  slot %llu: back-substituted inverse is wrong\n", (unsigned long long)j); }
                        (kind == PAIR_ADD ? nadd : ndbl)++;
                    }
                    a = pair_sum<F>(kind, a.x, a.y, b.x, b.y, inv);
                }
            }
            np[o] = a; nk[o] = keys[s];
        }
    }
    keys.swap(nk); pts.swap(np);
}

template <class F> static int check(const char* name, const Affine<F>& g) {
    const uint32_t NB = 97;
    std::vector<Affine<F>> base(64);
    for (size_t i = 0; i < base.size(); i++) base[i] = mul_small(g, 1000 + 7919 * (uint32_t)i);
    Affine<F> inf; inf.x = F::zero(); inf.y = F::zero();
    std::vector<uint32_t> keys; std::vector<Affine<F>> pts;
    auto push = [&](uint32_t k, const Affine<F>& p) { keys.push_back(k); pts.push_back(p); };
    for (uint32_t b = 0; b < NB; b++) {
        const int len = b % 11 == 3 ? 0 : 1 + (int)(rnd() % 9);               // odd and even runs, some empty buckets
        for (int e = 0; e < len; e++) {
            Affine<F> p = base[rnd() % base.size()];
            if (rnd() % 2) p.y = F::neg(p.y);                                  // signed digits
            if (rnd() % 23 == 0) p = inf;                                      // bases at infinity
            push(b, p);
        }
        if (b % 7 == 2) { const Affine<F> p = base[b % base.size()]; for (int e = 0; e < 8; e++) push(b, p); }      // P + P, 2P + 2P, 4P + 4P
        if (b % 9 == 4) { Affine<F> p = base[(b + 1) % base.size()], q = p; q.y = F::neg(q.y); push(b, p); push(b, q); }   // P + (-P)
        if (b % 13 == 5) { push(b, inf); push(b, base[3]); }                  // infinity first in a pair
    }
    const std::vector<Affine<F>> want = bucket_sums(keys, pts, NB);
    int bad = 0, nadd = 0, ndbl = 0;
    const uint64_t n0 = keys.size();
    const uint64_t Ts[] = {3, 128, 5, 1};
    for (int r = 0; r < 4; r++) {
        const uint64_t T = Ts[r], J = (keys.size() + 1) / 2;
        const uint32_t K = (uint32_t)((J + T - 1) / T);
        round_model<F>(keys, pts, T, K, nadd, ndbl);
        for (size_t i = 1; i < keys.size(); i++) if (keys[i - 1] > keys[i]) { bad++; printf("%s: round %d: list not sorted at %zu\n", name, r, i); break; }
        const std::vector<Affine<F>> got = bucket_sums(keys, pts, NB);
        for (uint32_t b = 0; b < NB; b++) if (!same(got[b], want[b])) { bad++; if (bad < 5) printf("%s: round %d: bucket %u differs\n", name, r, b); }
    }
    printf("%s: %s (%llu entries -> %zu after 4 rounds, %d additions, %d doublings)\n", name, bad ? "FAIL" : "ok",
           (unsigned long long)n0, keys.size(), nadd, ndbl);
    if (!ndbl) { bad++; printf("%s: no doubling exercised\n", name); }
    return bad;
}

int main() {
    int bad = 0;
    {
        Affine<Fp<BnFq>> g; g.x = from_hex<BnFq>("1"); g.y = from_hex<BnFq>("2");
        bad += check<Fp<BnFq>>("BN254 G1", g);
        Affine<Fp2<BnFq>> h;
        h.x.a = from_hex<BnFq>("1800deef121f1e76426a00665e5c4479674322d4f75edadd46debd5cd992f6ed");
        h.x.b = from_hex<BnFq>("198e9393920d483a7260bfb731fb5d25f1aa493335a9e71297e485b7aef312c2");
        h.y.a = from_hex<BnFq>("12c85ea5db8c6deb4aab71808dcb408fe3d1e7690c43d37b4ce6cc0166fa7daa");
        h.y.b = from_hex<BnFq>("090689d0585ff075ec9e99ad690c3395bc4b313370b38ef355acdadcd122975b");
        bad += check<Fp2<BnFq>>("BN254 G2", h);
    }
    {
        Affine<Fp<BlsFq>> g;
        g.x = from_hex<BlsFq>("17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb");
        g.y = from_hex<BlsFq>("08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1");
        bad += check<Fp<BlsFq>>("BLS12-381 G1", g);
        Affine<Fp2<BlsFq>> h;
        h.x.a = from_hex<BlsFq>("024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8");
        h.x.b = from_hex<BlsFq>("13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e");
        h.y.a = from_hex<BlsFq>("0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801");
        h.y.b = from_hex<BlsFq>("0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be");
        bad += check<Fp2<BlsFq>>("BLS12-381 G2", h);
    }
    bad += g_bad_inverse;
    printf(bad ? "BATCH AFFINE CHECK FAILED\n" : "BATCH AFFINE CHECK PASSED\n");
    return bad ? 1 : 0;
}
