// Host emulation library of the kernels (emu_lib.cpp, unchanged) plus one probe of the discrete auxiliary mode's workspace layout,
// for the stage-level tests of tests/test_discrete_grad.py.  TEST INFRASTRUCTURE ONLY.
#include "emu_lib.cpp"

// Byte offsets of the discrete-mode stage arrays in the workspace (which: 0 = Hth, 1 = E).
extern "C" CPDP_API size_t cpdp_emu_disc_offset(int B, int N, int S, int which) {
    char* const base = reinterpret_cast<char*>(static_cast<uintptr_t>(256));
    const CPDP_NS::WsLayout w = CPDP_NS::ws_carve(base, B, N, S);
    return (size_t)(reinterpret_cast<char*>(which == 0 ? w.disc.Hth : w.disc.E) - base);
}
