"""CPU-side support of the pdata-bound tests: the thread-emulated kernel library (tests/emu/emu_lib.cpp) of a model whose bounds may
depend on its per-problem constants, built with the model header and the companion header (bound Jacobians included) exactly as
COCSys.build generates them.  TEST INFRASTRUCTURE — the product never imports this."""
import hashlib
import os

import lfsd_b200  # noqa: F401
from lfsd_b200 import _capi, codegen, standard
from tests.emu.build_emu import build
from tests.emu.support import NumpyMem, _BUILD

_HERE = os.path.dirname(os.path.abspath(__file__))


def emu_pdb_from(oc, name, tsan=False):
    """Binds COCSys `oc` to the host-emulated kernels of its generated headers (model + pdata companion); returns `oc`."""
    args = (oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar)
    tv = getattr(oc, 'time', None)
    text, _ = codegen.generate_model_header(name, *args, time=tv, bounds=oc._bounds())
    pd_text, _ = codegen.generate_pdata_header(name, *args, time=tv, bounds=oc._bounds())
    src = "".join(open(os.path.join(_capi.CSRC, f)).read() for f in sorted(os.listdir(_capi.CSRC))
                  if os.path.isfile(os.path.join(_capi.CSRC, f)))
    src += open(os.path.join(_HERE, "emu_lib.cpp")).read()
    tag = hashlib.sha1((text + pd_text + src + str(tsan)).encode()).hexdigest()[:12]
    os.makedirs(_BUILD, exist_ok=True)
    hdr = os.path.join(_BUILD, "model_%s_%s.cuh" % (name, tag))
    pd_hdr = os.path.join(_BUILD, "model_%s_%s_pd.cuh" % (name, tag))
    so = os.path.join(_BUILD, "libemupdb_%s_%s.so" % (name, tag))
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        with open(pd_hdr, "w") as f:
            f.write(pd_text)
        tmp = "%s.tmp%d" % (so, os.getpid())
        build(hdr, tmp, tsan=tsan, ns="cpdp_emupdb_" + name, extra=["-DCPDP_WITH_BDF", "-DCPDP_PD_HEADER=\"%s\"" % pd_hdr])
        os.replace(tmp, so)
    oc._lib = _capi.CpdpLib(so)
    oc._mem = NumpyMem()
    return oc


def emu_pdb_oc(name, tsan=False, **kw):
    """COCSys of standard.PD_BOUNDED (or standard.BOUNDED) model `name` bound to the host-emulated kernels."""
    fn = standard.PD_BOUNDED.get(name) or standard.BOUNDED[name]
    return emu_pdb_from(fn(**kw), name, tsan=tsan)
