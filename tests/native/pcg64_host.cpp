// TEST HARNESS (not part of the product): compiles the SHIPPED PCG64 code of csrc/mpcb_pcg64.cuh for the host with g++,
// so that tests/test_pcg64_on_host.py can compare it with numpy's Generator(PCG64) without a GPU.  Every draw entry
// works in place on one record rec[6] = state hi/lo, inc hi/lo, has_uint32, uinteger.
#include "mpcb_pcg64.cuh"

extern "C" void mpcb_test_pcg64_seed(const unsigned *entropy, int E, const unsigned *spawn, int K,
                                     unsigned long long *rec) {
    mpcb::pcg64_seed(entropy, E, spawn, K, rec);
}

// ops[i] = 0: random() into val[i]; ops[i] = 1: integers(lo[i], hi[i]) into val[i] (as a double: the ranges are small)
extern "C" void mpcb_test_pcg64_draws(unsigned long long *rec, long long n, const int *ops, const long long *lo,
                                      const long long *hi, double *val) {
    mpcb::Pcg64 g = mpcb::pcg64_load(rec);
    for (long long i = 0; i < n; ++i)
        val[i] = ops[i] == 0 ? mpcb::pcg64_random(g) : (double)mpcb::pcg64_integers(g, lo[i], hi[i]);
    mpcb::pcg64_store(g, rec);
}

// the draws of one tick of the device loop: velocity first, then beta
extern "C" void mpcb_test_pcg64_actuators(unsigned long long *rec, long long n, const double *v_ref,
                                          const double *beta_ref, double *v_out, double *beta_out) {
    mpcb::Pcg64 g = mpcb::pcg64_load(rec);
    for (long long i = 0; i < n; ++i) {
        v_out[i] = mpcb::actual_velocity(v_ref[i], g);
        beta_out[i] = mpcb::actual_beta(beta_ref[i], g);
    }
    mpcb::pcg64_store(g, rec);
}
