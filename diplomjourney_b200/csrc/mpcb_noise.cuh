// mpcb_noise.cuh -- the actuator disturbance of the online controller's "actual" run (math_model_tree.py:259-275), drawn
// from numpy's legacy RandomState stream bit for bit, so a device run reproduces the reference's seeded runs.  Plain
// host/device code: the CPU test-suite compiles exactly this with g++ and compares it with np.random.RandomState
// (tests/test_noise_on_host.py).
//
// Generator state = what RandomState.get_state() hands out: st[0..623] = key, st[624] = pos (624 right after seeding,
// so the first draw twists).  The draws continue any state where it stands, mid-stream ones included; mt_seed and
// mt_seed_by_array build the state RandomState(int) and RandomState(array) start from (tests/test_seed_on_host.py).
#pragma once
#include "mpcb_types.cuh"

namespace mpcb {

constexpr int kMtN = 624, kMtM = 397;
constexpr int kMtWords = kMtN + 1;     // key + pos, the per-robot record of mpcb_held_closed_loop_actual_host

MPCB_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

// RandomState(s) / np.random.seed(s): numpy's mt19937_seed, all arithmetic mod 2^32
MPCB_HD void mt_seed(unsigned *st, unsigned s) {
    for (int i = 0; i < kMtN; ++i) {
        st[i] = s;
        s = 1812433253u * (s ^ (s >> 30)) + (unsigned)i + 1u;
    }
    st[kMtN] = kMtN;
}

// RandomState(key) for a 1-D key of K >= 1 words: numpy's mt19937_init_by_array.  RandomState(5) and RandomState([5])
// are different streams.  `prev` is mt[i - 1]; on the wrap of i it is mt[623], which is also the new mt[0].
MPCB_HD void mt_seed_by_array(unsigned *st, const unsigned *key, int K) {
    mt_seed(st, 19650218u);
    int i = 1, j = 0;
    unsigned prev = st[0];
    for (int k = K > kMtN ? K : kMtN; k > 0; --k) {
        prev = st[i] = (st[i] ^ ((prev ^ (prev >> 30)) * 1664525u)) + key[j] + (unsigned)j;
        if (++i >= kMtN) { st[0] = prev; i = 1; }
        if (++j >= K) j = 0;
    }
    for (int k = kMtN - 1; k > 0; --k) {
        prev = st[i] = (st[i] ^ ((prev ^ (prev >> 30)) * 1566083941u)) - (unsigned)i;
        if (++i >= kMtN) { st[0] = prev; i = 1; }
    }
    st[0] = 0x80000000u;        // the most significant bit set: the state is never all zero
    st[kMtN] = kMtN;
}

// the standard MT19937 twist of all 624 words; pos := 0.  Not inlined: it runs once per 312+ draws, and inlined into the
// loop kernel it made ptxas spill
static MPCB_HD_NOINLINE void mt_twist(unsigned *st) {
    const unsigned upper = 0x80000000u, lower = 0x7fffffffu, matrix_a = 0x9908b0dfu;
    int i = 0;
    for (; i < kMtN - kMtM; ++i) {
        const unsigned y = (st[i] & upper) | (st[i + 1] & lower);
        st[i] = st[i + kMtM] ^ (y >> 1) ^ ((0u - (y & 1u)) & matrix_a);
    }
    for (; i < kMtN - 1; ++i) {
        const unsigned y = (st[i] & upper) | (st[i + 1] & lower);
        st[i] = st[i + kMtM - kMtN] ^ (y >> 1) ^ ((0u - (y & 1u)) & matrix_a);
    }
    const unsigned y = (st[kMtN - 1] & upper) | (st[0] & lower);
    st[kMtN - 1] = st[kMtM - 1] ^ (y >> 1) ^ ((0u - (y & 1u)) & matrix_a);
    st[kMtN] = 0;
}

// one tempered 32-bit word
MPCB_HD unsigned mt_next_u32(unsigned *st) {
    if (st[kMtN] >= (unsigned)kMtN) mt_twist(st);
    unsigned y = st[st[kMtN]++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// RandomState.random() / random_sample(): 53 bits from two words
MPCB_HD double np_random_sample(unsigned *st) {
    const unsigned a = mt_next_u32(st) >> 5;
    const unsigned b = mt_next_u32(st) >> 6;
    return ddiv(dadd(dmul((double)a, 67108864.0), (double)b), 9007199254740992.0);
}

// RandomState.randint(lo, hi), hi exclusive, hi - lo <= 2^31: masked rejection, one word per attempt (so a draw takes a
// varying number of words; none at all when the range holds one value)
MPCB_HD int np_randint_masked(unsigned *st, int lo, int hi) {
    const unsigned rng = (unsigned)(hi - 1 - lo);
    if (rng == 0) return lo;
    unsigned mask = rng;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    unsigned v;
    do v = mt_next_u32(st) & mask; while (v > rng);
    return lo + (int)v;
}

// get_actual_velocity (math_model_tree.py:259-275): one random(); below 0.7 a jitter of randint(0, 5) / 1000 under
// 0.4 m/s, else randint(-100, 10) / 1000
MPCB_HD double actual_velocity(double v_ref, unsigned *st) {
    if (!(np_random_sample(st) < 0.7)) return v_ref;
    const int k = v_ref < 0.4 ? np_randint_masked(st, 0, 5) : np_randint_masked(st, -100, 10);
    return dadd(v_ref, ddiv((double)k, 1000.0));
}

// get_actual_beta_angle (math_model_tree.py:259-275): one random(); below 0.7 beta_ref + radians(randint(-5, 5))
MPCB_HD double actual_beta(double beta_ref, unsigned *st) {
    if (!(np_random_sample(st) < 0.7)) return beta_ref;
    const int k = np_randint_masked(st, -5, 5);
    return dadd(beta_ref, dmul((double)k, 3.141592653589793 / 180.0));     // math.radians(k) == k * (pi / 180)
}

}  // namespace mpcb
