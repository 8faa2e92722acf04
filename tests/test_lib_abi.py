"""CPU-side checks of the drop-in boundary: libegot2.so loads and exports exactly the entry points that
include/egot2.h declares (no compute is launched here)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "egot2.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(egot2_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def built():
    from egot2_b200 import build
    return build.build()


def test_header_symbols_are_exported_and_bound(built):
    from egot2_b200 import _lib
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/egot2.h but not exported by libegot2.so"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in egot2_b200/_lib.py"
    for name in _lib.SIGNATURES:
        assert name in declared, f"{name} bound in _lib.py but not declared in include/egot2.h"
    assert b"sm_100a" in lib.egot2_version()


def test_struct_layouts_match_header(built):
    """sizeof() of every ctypes mirror must equal the C struct (checked through a tiny compiled probe)."""
    import ctypes as C
    import subprocess
    import tempfile
    from egot2_b200 import _lib
    names = {"egot2_embed_desc": _lib.EmbedDesc, "egot2_embed_in": _lib.EmbedIn, "egot2_embed_out": _lib.EmbedOut,
             "egot2_embed_grads": _lib.EmbedGrads, "egot2_layer_desc": _lib.LayerDesc,
             "egot2_layer_params": _lib.LayerParams, "egot2_layer_grads": _lib.LayerGrads,
             "egot2_layer_saved": _lib.LayerSaved, "egot2_head_desc": _lib.HeadDesc, "egot2_head_in": _lib.HeadIn,
             "egot2_head_out": _lib.HeadOut, "egot2_head_grads": _lib.HeadGrads,
             "egot2_decoder_desc": _lib.DecoderDesc, "egot2_decoder_params": _lib.DecoderParams,
             "egot2_decoder_grads": _lib.DecoderGrads, "egot2_decoder_saved": _lib.DecoderSaved,
             "egot2_vit_desc": _lib.VitDesc, "egot2_vit_params": _lib.VitParams, "egot2_vit_grads": _lib.VitGrads,
             "egot2_vit_saved": _lib.VitSaved, "egot2_dp_desc": _lib.DpDesc}
    # (struct, field) pairs whose byte offsets are compared as well: the last fields of the descriptors that grew
    offsets = [("egot2_embed_desc", "seed"), ("egot2_embed_desc", "no_ln"), ("egot2_embed_desc", "feat_drop_tokens"), ("egot2_vit_desc", "ln_eps"),
               ("egot2_vit_saved", "act"), ("egot2_decoder_desc", "seed"), ("egot2_head_desc", "seed"),
               ("egot2_dp_desc", "off_flags"), ("egot2_dp_desc", "exp_avg"), ("egot2_dp_desc", "step_dev"), ("egot2_dp_desc", "zero_grads_remote")]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));' for n in names) + "".join(
        f'printf("{n}.{f} %zu\\n", offsetof({n}, {f}));' for n, f in offsets) + "return 0;}"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, size = line.split()
        if "." in n:
            st, f = n.split(".")
            assert getattr(names[st], f).offset == int(size), f"{n}: ctypes offset {getattr(names[st], f).offset} != C {size}"
        else:
            assert C.sizeof(names[n]) == int(size), f"{n}: ctypes {C.sizeof(names[n])} != C {size}"


def test_no_fallback_without_cuda():
    """Without a CUDA device the engine refuses to run; checked in a child process that sees no device, so that a machine
    with a GPU checks it too."""
    import subprocess
    import sys
    code = ("import pytest, torch\n"
            "from egot2_b200 import _lib, specs\n"
            "from egot2_b200.engine import TranslatorEngine\n"
            "assert not torch.cuda.is_available()\n"
            "with pytest.raises(_lib.Egot2Error):\n"
            "    TranslatorEngine(specs.hhi_ttm_spec(), 'cpu')\n")
    flags = ["-s"] if sys.flags.no_user_site else []
    subprocess.run([sys.executable, *flags, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), check=True)
