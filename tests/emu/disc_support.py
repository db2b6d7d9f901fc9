"""CPU-side support of the discrete-mode tests: the thread-emulated kernel library of tests/emu/emu_lib.cpp extended by
tests/emu/emu_disc_lib.cpp with a probe of the workspace layout (byte offsets of the mode-2 stage arrays).
TEST INFRASTRUCTURE — the product never imports this."""
import hashlib
import os
import subprocess

from lfsd_b200 import _capi, codegen, standard
from tests.emu.build_emu import CSRC
from tests.emu.support import NumpyMem, _BUILD

_HERE = os.path.dirname(os.path.abspath(__file__))


def emu_disc_oc(name, **kw):
    """COCSys for standard model `name` bound to the emulated kernels plus cpdp_emu_disc_offset(B, N, S, which)."""
    oc = (standard.STANDARD.get(name) or standard.VARIANTS[name])(**kw)
    text, info = codegen.generate_model_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost,
                                               oc.final_cost, oc.pvar, time=getattr(oc, 'time', None))
    os.makedirs(_BUILD, exist_ok=True)
    src = ""
    for fn in sorted(os.listdir(_capi.CSRC)):
        p = os.path.join(_capi.CSRC, fn)
        if os.path.isfile(p):
            src += open(p).read()
    for fn in ("emu_lib.cpp", "emu_disc_lib.cpp"):
        src += open(os.path.join(_HERE, fn)).read()
    tag = hashlib.sha1((text + src).encode()).hexdigest()[:12]
    hdr = os.path.join(_BUILD, "model_%s_%s.cuh" % (name, tag))
    so = os.path.join(_BUILD, "libemudisc_%s_%s.so" % (name, tag))
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        tmp = "%s.tmp%d" % (so, os.getpid())
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-g", "-fPIC", "-shared", "-pthread", "-fvisibility=hidden",
                               "-fno-gnu-unique", "-DCPDP_NS=cpdp_emudisc_" + name, "-I", CSRC,
                               "-DCPDP_MODEL_HEADER_PORT=\"cpdp_port.h\"", "-DCPDP_MODEL_HEADER=\"%s\"" % hdr, "-DCPDP_WITH_BDF",
                               os.path.join(_HERE, "emu_disc_lib.cpp"), "-o", tmp])
        os.replace(tmp, so)
    oc._lib = _capi.CpdpLib(so)
    oc._mem = NumpyMem()
    return oc
