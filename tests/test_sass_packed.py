"""CPU tier: the fp32 site arithmetic of the shipped build runs on the paired FP32 pipe (cuobjdump / ptxas log of the build's
sm_100a objects; nothing is executed).  The headline kernel -- fp32 recon-12 Wilson interior, no dagger, no xpay -- does its
complex arithmetic as FFMA2 / FADD2 / FMUL2 on (re, im) register pairs: 976 SASS instructions per thread against 1 520 with
scalar FFMA / FADD / FMUL (B2_PACKED_F32=0), and no more spilled bytes than the scalar build (4)."""
import functools
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "quda_b200", "csrc", "_obj")
HEADLINE = "b200::dslash_interior_kernel<b200::PrecF32, 12, false, false, (b200::OpType)0, false>"

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(os.path.join(OBJ, "inst_f32.o")),
                                reason="needs cuobjdump and the build's object files (__graft_entry__.build())")


def _demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


@functools.lru_cache(maxsize=None)
def _mnemonics(obj):
    """{demangled function: [mnemonic]} of one object file"""
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(OBJ, obj)], capture_output=True, text=True, errors="replace").stdout
    funs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funs[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and cur:
            funs[cur].append(m.group(1).split(".")[0])
    names = _demangle(list(funs))
    return {names[k]: v for k, v in funs.items()}


def _kernel(obj, prefix):
    hits = [v for k, v in _mnemonics(obj).items() if k.startswith("void " + prefix)]
    assert len(hits) == 1, prefix
    return hits[0]


@pytest.mark.parametrize("recon", [12, 18])
def test_fp32_wilson_interior_runs_on_paired_fp32(recon):
    ins = _kernel("inst_f32.o", f"b200::dslash_interior_kernel<b200::PrecF32, {recon}, false, false, (b200::OpType)0, false>")
    assert ins.count("FFMA2") >= 300
    assert "FADD2" in ins
    scalar = sum(ins.count(k) for k in ("FFMA", "FADD", "FMUL"))
    assert scalar == 0, f"{scalar} scalar fp32 instructions left in the stencil"


def test_headline_kernel_instruction_count():
    assert len(_kernel("inst_f32.o", HEADLINE)) <= 1050


def test_headline_kernel_spills_no_more_than_the_scalar_build():
    log = os.path.join(OBJ, "inst_f32.ptxas.log")
    if not os.path.exists(log):
        pytest.skip("no ptxas log next to the objects")
    spills, name = {}, None
    for line in open(log, errors="replace"):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            spills[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    hits = [spills[k] for k, v in _demangle(list(spills)).items() if v.startswith("void " + HEADLINE)]
    assert len(hits) == 1
    st, ld = hits[0]
    assert st <= 4 and ld <= 4, (st, ld)
