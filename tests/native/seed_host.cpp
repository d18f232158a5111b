// TEST HARNESS (not part of the product): compiles the SHIPPED seeding code of csrc/mpcb_noise.cuh for the host with
// g++, so that tests/test_seed_on_host.py can compare it with numpy's RandomState(seed) without a GPU.  Every entry
// writes one generator record st[625] = key[624], pos.
#include "mpcb_noise.cuh"

extern "C" void mpcb_test_mt_seed(unsigned *st, unsigned s) { mpcb::mt_seed(st, s); }

extern "C" void mpcb_test_mt_seed_by_array(unsigned *st, const unsigned *key, int K) {
    mpcb::mt_seed_by_array(st, key, K);
}
