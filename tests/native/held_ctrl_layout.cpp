// Layout of mpcb_held_ctrl as a C++ compiler lays it out from the public header: sizeof, alignof and every field's
// offset and size, one "name offset size" line each (tests/test_held_ctrl_on_host.py compares them with the ctypes
// mirror in diplomjourney_b200/_native.py).
#include <cstddef>
#include <cstdio>

#include "mpcb200.h"

#define FIELD(f) std::printf(#f " %zu %zu\n", offsetof(mpcb_held_ctrl, f), sizeof(((mpcb_held_ctrl *)0)->f))

int main() {
    std::printf("sizeof %zu\nalignof %zu\n", sizeof(mpcb_held_ctrl), alignof(mpcb_held_ctrl));
    FIELD(pose); FIELD(line); FIELD(threshold); FIELD(prev); FIELD(opt); FIELD(command);
    FIELD(slow_steps); FIELD(m); FIELD(ticks); FIELD(status); FIELD(recursive); FIELD(have_traj); FIELD(pending);
    FIELD(reserved);
    std::printf("MPCB_LOOP_RUNNING %d 0\n", MPCB_LOOP_RUNNING);
    return 0;
}
