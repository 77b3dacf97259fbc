"""integration/mcs_shim.jl cannot be executed here (no Julia in the image): check it structurally instead.  The struct
definitions are parsed and laid out with C rules; names, order, offsets and sizes must equal the ctypes mirror that every
GPU test runs through (abi.py), which in turn is checked against the library's own sizeof (mcs_abi_sizes).  Also: every
symbol the shim ccalls is declared in include/mcs.h, and the recorder's patch anchors exist in the reference sources when
MCS_REFERENCE_SRC names them."""
import ctypes as C
import os
import re

import pytest

from mcs_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "integration", "mcs_shim.jl")

_SIZES = {"Int32": 4, "UInt32": 4, "Int64": 8, "UInt64": 8, "Float64": 8, "UInt8": 1}


def _julia_type(t):
    """(size, align, count) of a Julia field type as C lays it out."""
    t = t.strip()
    if t.startswith("Ptr{"):
        return 8, 8
    m = re.fullmatch(r"NTuple\{\s*(\d+)\s*,\s*(\w+)\s*\}", t)
    if m:
        return int(m.group(1)) * _SIZES[m.group(2)], _SIZES[m.group(2)]
    return _SIZES[t], _SIZES[t]


def parse_structs(text):
    out = {}
    for m in re.finditer(r"^struct (\w+)\n(.*?)^end", text, re.S | re.M):
        fields = []
        for line in m.group(2).splitlines():
            line = line.split("#")[0].strip()
            for part in line.split(";"):
                part = part.strip()
                if "::" in part:
                    nm, ty = part.split("::")
                    fields.append((nm.strip(), ty.strip()))
        out[m.group(1)] = fields
    return out


def c_layout(fields):
    off, maxal, res = 0, 1, []
    for nm, ty in fields:
        sz, al = _julia_type(ty)
        off = (off + al - 1) // al * al
        res.append((nm, off, sz))
        off += sz
        maxal = max(maxal, al)
    return res, (off + maxal - 1) // maxal * maxal


@pytest.mark.parametrize("name", ["McsConfig", "McsSpecies", "McsTallies", "McsPopulation", "McsInjection", "McsTraceRec", "McsTiming", "McsThermoIn"])
def test_struct_layout_matches_ctypes(name):
    structs = parse_structs(open(SHIM).read())
    assert name in structs, f"{name} missing from mcs_shim.jl"
    lay, size = c_layout(structs[name])
    ct = getattr(abi, name)
    want = [(f[0], getattr(ct, f[0]).offset, getattr(ct, f[0]).size) for f in ct._fields_]
    assert lay == want
    assert size == C.sizeof(ct)


def test_every_ccall_symbol_is_declared():
    text = open(SHIM).read()
    header = open(os.path.join(ROOT, "include", "mcs.h")).read()
    syms = set(re.findall(r"\(:(mcs_\w+), LIBMCS\)", text))
    assert {"mcs_create", "mcs_set_profile", "mcs_begin_ion", "mcs_run_ion", "mcs_end_ion", "mcs_abi_sizes"} <= syms
    for s in syms:
        assert re.search(rf"\b{s}\s*\(", header), f"{s} is not declared in include/mcs.h"
        assert s in abi.ABI_SYMBOLS


def test_recorder_anchors_exist_in_reference():
    """MCS_REFERENCE_SRC: the src/ directory of a MonteCarloScattering.jl checkout, whose sources this repository does not
    contain."""
    ref = os.environ.get("MCS_REFERENCE_SRC", "")
    if not os.path.isdir(ref):
        pytest.skip("MCS_REFERENCE_SRC does not name the src/ directory of a MonteCarloScattering.jl checkout")
    rec = open(os.path.join(ROOT, "tools", "record_reference.jl")).read()
    src = {"particle_loop.jl": open(os.path.join(ref, "particle_loop.jl")).read(),
           "main_loops.jl": open(os.path.join(ref, "main_loops.jl")).read()}
    anchors = {
        "particle_loop.jl": ["rng = Random.Xoshiro(iseed_mod)", "        # If particle escaped downstream, handle final calculations here",
                             "    end # loop_helix\n"],
        "main_loops.jl": ["            weight_running = weight_in[1]\n", "                for i_prt in 1:n_pts_use # loop_pt\n",
                          "                # Conclusion of particle loop\n", "            # Conclusion of pcuts loop\n"],
    }
    for f, lst in anchors.items():
        for a in lst:
            assert src[f].count(a) == 1, (f, a)
            assert a.strip("\n") .strip() in rec or a in rec
