"""CPU-side support of the bound tests: the thread-emulated kernel library (tests/emu/emu_lib.cpp) for a box-bounded model,
whose generated header carries the bounds.  TEST INFRASTRUCTURE — the product never imports this."""
import hashlib
import os

import lfsd_b200  # noqa: F401
from lfsd_b200 import _capi, codegen, standard
from tests.emu.build_emu import build
from tests.emu.support import NumpyMem, _BUILD

_HERE = os.path.dirname(os.path.abspath(__file__))


def emu_from(oc, name, tsan=False):
    """Binds COCSys `oc` (bounded or not) to the host-emulated kernels of its generated header; returns `oc`."""
    text, _ = codegen.generate_model_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar,
                                            time=getattr(oc, 'time', None), bounds=oc._bounds())
    src = "".join(open(os.path.join(_capi.CSRC, f)).read() for f in sorted(os.listdir(_capi.CSRC))
                  if os.path.isfile(os.path.join(_capi.CSRC, f)))
    src += open(os.path.join(_HERE, "emu_lib.cpp")).read()
    tag = hashlib.sha1((text + src + str(tsan)).encode()).hexdigest()[:12]
    os.makedirs(_BUILD, exist_ok=True)
    hdr = os.path.join(_BUILD, "model_%s_%s.cuh" % (name, tag))
    so = os.path.join(_BUILD, "libemu_%s_%s.so" % (name, tag))
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        build(hdr, so, tsan=tsan, ns="cpdp_emu_" + name, extra=["-DCPDP_WITH_BDF"])
    oc._lib = _capi.CpdpLib(so)
    oc._mem = NumpyMem()
    return oc


def emu_bounded_oc(name, tsan=False, **kw):
    """COCSys of standard.BOUNDED model `name` bound to the host-emulated kernels."""
    return emu_from(standard.BOUNDED[name](**kw), name, tsan=tsan)
