// mpcb_pcg64.cuh -- the actuator disturbance of the "actual" run drawn from numpy's Generator(PCG64) stream bit for bit,
// beside the legacy RandomState stream of mpcb_noise.cuh.  Plain host/device code: the CPU test-suite compiles exactly
// this with g++ and compares it with np.random.Generator (tests/test_pcg64_on_host.py).
//
// Generator state = what Generator(PCG64).bit_generator.state hands out, as one record of kPcgWords u64 words:
//   [0] state >> 64, [1] state mod 2^64, [2] inc >> 64, [3] inc mod 2^64, [4] has_uint32 (0/1), [5] uinteger (< 2^32)
// One step is state = state * M + inc (mod 2^128), and the step comes before the output (XSL-RR).  The 32-bit draws
// (integers() on ranges below 2^32) hand out the low half of a 64-bit output and keep the high half in
// (has_uint32, uinteger) for the next 32-bit draw, across calls: the buffer is part of the state.
// pcg64_seed builds the record default_rng(SeedSequence(entropy, spawn_key)) starts from.
#pragma once
#include "mpcb_noise.cuh"

namespace mpcb {

constexpr int kPcgWords = 6;    // the per-robot record of mpcb_held_closed_loop_pcg64_host
constexpr unsigned long long kPcgMultHi = 2549297995355413924ull, kPcgMultLo = 4865540595714422341ull;

struct Pcg64 {
    unsigned long long hi, lo, inc_hi, inc_lo;
    unsigned has_uint32, uinteger;
};

MPCB_HD Pcg64 pcg64_load(const unsigned long long *r) {
    Pcg64 g;
    g.hi = r[0]; g.lo = r[1]; g.inc_hi = r[2]; g.inc_lo = r[3];
    g.has_uint32 = (unsigned)r[4]; g.uinteger = (unsigned)r[5];
    return g;
}

MPCB_HD void pcg64_store(const Pcg64 &g, unsigned long long *r) {
    r[0] = g.hi; r[1] = g.lo; r[2] = g.inc_hi; r[3] = g.inc_lo; r[4] = g.has_uint32; r[5] = g.uinteger;
}

// the upper 64 bits of a 64 x 64-bit product: the one primitive of the 128-bit arithmetic that differs by target
MPCB_HD unsigned long long umulhi64(unsigned long long a, unsigned long long b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (unsigned long long)(((unsigned __int128)a * b) >> 64);
#endif
}

// (hi, lo) := (hi, lo) * M + (inc_hi, inc_lo)  mod 2^128
MPCB_HD void pcg64_step(unsigned long long &hi, unsigned long long &lo, unsigned long long inc_hi,
                        unsigned long long inc_lo) {
    const unsigned long long phi = umulhi64(lo, kPcgMultLo) + hi * kPcgMultLo + lo * kPcgMultHi;
    const unsigned long long plo = lo * kPcgMultLo;
    lo = plo + inc_lo;
    hi = phi + inc_hi + (lo < plo ? 1ull : 0ull);
}

// XSL-RR: (hi ^ lo) rotated right by the top six bits of hi
MPCB_HD unsigned long long pcg64_output(unsigned long long hi, unsigned long long lo) {
    const unsigned long long x = hi ^ lo;
    const unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}

MPCB_HD unsigned long long pcg64_next64(Pcg64 &g) {
    pcg64_step(g.hi, g.lo, g.inc_hi, g.inc_lo);
    return pcg64_output(g.hi, g.lo);
}

// the buffered upper half if there is one, else the low half of a new output (its upper half buffered)
MPCB_HD unsigned pcg64_next32(Pcg64 &g) {
    if (g.has_uint32) { g.has_uint32 = 0; return g.uinteger; }
    const unsigned long long v = pcg64_next64(g);
    g.has_uint32 = 1;
    g.uinteger = (unsigned)(v >> 32);
    return (unsigned)v;
}

// Generator.random(): 53 bits of one 64-bit output; the 32-bit buffer is left as it is
MPCB_HD double pcg64_random(Pcg64 &g) {
    return dmul((double)(pcg64_next64(g) >> 11), 1.0 / 9007199254740992.0);
}

// Generator.integers(lo, hi), hi exclusive, hi - lo <= 2^32 - 1: numpy's buffered_bounded_lemire_uint32 on the 32-bit
// draws (one word per attempt; none when the range holds one value)
MPCB_HD long long pcg64_integers(Pcg64 &g, long long lo, long long hi) {
    const unsigned rng = (unsigned)(hi - 1 - lo);
    if (rng == 0) return lo;
    const unsigned rng_excl = rng + 1u;
    unsigned long long m = (unsigned long long)pcg64_next32(g) * rng_excl;
    unsigned left = (unsigned)m;
    if (left < rng_excl) {
        const unsigned threshold = (0xffffffffu - rng) % rng_excl;
        while (left < threshold) {
            m = (unsigned long long)pcg64_next32(g) * rng_excl;
            left = (unsigned)m;
        }
    }
    return lo + (long long)(m >> 32);
}

// get_actual_velocity with a Generator (math_model_tree.py:259-275): one random(); below 0.7 a jitter of
// integers(0, 5) / 1000 under 0.4 m/s, else integers(-100, 10) / 1000 -- the draw order of the MT19937 version
MPCB_HD double actual_velocity(double v_ref, Pcg64 &g) {
    if (!(pcg64_random(g) < 0.7)) return v_ref;
    const long long k = v_ref < 0.4 ? pcg64_integers(g, 0, 5) : pcg64_integers(g, -100, 10);
    return dadd(v_ref, ddiv((double)k, 1000.0));
}

// get_actual_beta_angle with a Generator: one random(); below 0.7 beta_ref + radians(integers(-5, 5))
MPCB_HD double actual_beta(double beta_ref, Pcg64 &g) {
    if (!(pcg64_random(g) < 0.7)) return beta_ref;
    const long long k = pcg64_integers(g, -5, 5);
    return dadd(beta_ref, dmul((double)k, 3.141592653589793 / 180.0));
}

// ---- seeding: numpy's SeedSequence (pool size 4, 32-bit words) and PCG64's use of generate_state(4, uint64)
constexpr unsigned kSsInitA = 0x43b0d7e5u, kSsMultA = 0x931e8875u, kSsInitB = 0x8b51f9ddu, kSsMultB = 0x58f38dedu;
constexpr unsigned kSsMixMultL = 0xca01f9ddu, kSsMixMultR = 0x4973f715u;
constexpr int kSsXshift = 16, kSsPool = 4;

MPCB_HD unsigned ss_hashmix(unsigned v, unsigned &hash_const) {
    v ^= hash_const;
    hash_const *= kSsMultA;
    v *= hash_const;
    return v ^ (v >> kSsXshift);
}

MPCB_HD unsigned ss_mix(unsigned x, unsigned y) {
    const unsigned r = kSsMixMultL * x - kSsMixMultR * y;
    return r ^ (r >> kSsXshift);
}

// word i of SeedSequence's assembled entropy: the entropy words, zero-padded to the pool size when there is a spawn key,
// then the spawn-key words
MPCB_HD unsigned ss_word(const unsigned *entropy, int E, const unsigned *spawn, int K, int i) {
    const int run = (K > 0 && E < kSsPool) ? kSsPool : E;
    if (i < E) return entropy[i];
    if (i < run) return 0u;
    return spawn[i - run];
}

// SeedSequence(entropy, spawn_key).generate_state(4, uint64) into w[4], then the PCG64 record seeded from it:
// initstate = w0 * 2^64 + w1, inc = ((w2 * 2^64 + w3) << 1) | 1, state = step(step(0) + initstate).  entropy[E] (E >= 1)
// are the entropy's little-endian 32-bit words (an integer expands into as many words as it needs, 0 into one word; a
// sequence of integers into the concatenation of theirs), spawn[K] the spawn key's words (K = 0: no spawn key).
MPCB_HD void pcg64_seed(const unsigned *entropy, int E, const unsigned *spawn, int K, unsigned long long *rec) {
    const int n = ((K > 0 && E < kSsPool) ? kSsPool : E) + K;
    unsigned pool[kSsPool];
    unsigned hc = kSsInitA;
    for (int i = 0; i < kSsPool; ++i) pool[i] = ss_hashmix(i < n ? ss_word(entropy, E, spawn, K, i) : 0u, hc);
    for (int s = 0; s < kSsPool; ++s)
        for (int d = 0; d < kSsPool; ++d)
            if (s != d) pool[d] = ss_mix(pool[d], ss_hashmix(pool[s], hc));
    for (int s = kSsPool; s < n; ++s) {
        const unsigned w = ss_word(entropy, E, spawn, K, s);
        for (int d = 0; d < kSsPool; ++d) pool[d] = ss_mix(pool[d], ss_hashmix(w, hc));
    }
    unsigned long long w[4];
    hc = kSsInitB;
    for (int i = 0; i < 8; ++i) {
        unsigned v = pool[i % kSsPool];
        v ^= hc;
        hc *= kSsMultB;
        v *= hc;
        v ^= v >> kSsXshift;
        if (i & 1) w[i >> 1] |= (unsigned long long)v << 32;
        else w[i >> 1] = v;
    }
    const unsigned long long inc_hi = (w[2] << 1) | (w[3] >> 63), inc_lo = (w[3] << 1) | 1ull;
    unsigned long long hi = 0, lo = 0;
    pcg64_step(hi, lo, inc_hi, inc_lo);
    const unsigned long long s_lo = lo + w[1];
    hi = hi + w[0] + (s_lo < lo ? 1ull : 0ull);
    lo = s_lo;
    pcg64_step(hi, lo, inc_hi, inc_lo);
    rec[0] = hi; rec[1] = lo; rec[2] = inc_hi; rec[3] = inc_lo; rec[4] = 0; rec[5] = 0;
}

}  // namespace mpcb
