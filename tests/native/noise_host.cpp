// TEST HARNESS (not part of the product): compiles the SHIPPED actuator-noise code of csrc/mpcb_noise.cuh for the host
// with g++, so that tests/test_noise_on_host.py can compare it with numpy's RandomState without a GPU.  Every entry
// works in place on one generator record st[625] = key[624], pos.
#include "mpcb_noise.cuh"

extern "C" void mpcb_test_mt_words(unsigned *st, long long n, unsigned *out) {
    for (long long i = 0; i < n; ++i) out[i] = mpcb::mt_next_u32(st);
}

extern "C" void mpcb_test_random_sample(unsigned *st, long long n, double *out) {
    for (long long i = 0; i < n; ++i) out[i] = mpcb::np_random_sample(st);
}

extern "C" void mpcb_test_randint(unsigned *st, int lo, int hi, long long n, long long *out) {
    for (long long i = 0; i < n; ++i) out[i] = mpcb::np_randint_masked(st, lo, hi);
}

// the draws of one tick of the device loop: velocity first, then beta
extern "C" void mpcb_test_actuators(unsigned *st, long long n, const double *v_ref, const double *beta_ref, double *v_out,
                                    double *beta_out) {
    for (long long i = 0; i < n; ++i) {
        v_out[i] = mpcb::actual_velocity(v_ref[i], st);
        beta_out[i] = mpcb::actual_beta(beta_ref[i], st);
    }
}
