"""CPU tier: static properties of the compiled sweep kernels (cuobjdump on the
built libpp2d.so; no GPU needed).  The fused kernel's speed depends on ptxas
seeing the marching loop as warp-uniform (DESIGN.md section 4): a divergence
guard (BRA.DIV) in front of the shuffles, or spills, cost 15-30 % and were
introduced silently more than once while the kernels were written (a
lane-0-only spin loop in the peer-to-peer variant was enough).  These checks
fail the build instead."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "path_planning_2d_b200", "libpp2d.so")

# T, CW, POLICY, P2P, LIN of the fused instantiations
FUSED = [(2, 2, p, q, l) for p in (0, 1) for q in (0, 1) for l in (0, 1)]


def mangled(t, cw, policy, p2p, lin):
    return (f"_ZN4pp2d16mdp_sweep_kernelILi{t}ELi{cw}ELb{policy}ELb{p2p}ELb{lin}EEEvNS_11SweepParamsE")


@pytest.fixture(scope="module")
def sass():
    from path_planning_2d_b200 import build
    # the toolkit that built the library also has cuobjdump, on PATH or not
    cuobjdump = (shutil.which("cuobjdump")
                 or os.path.join(os.path.dirname(build.NVCC), "cuobjdump"))
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    out = {}
    for key in FUSED:
        txt = subprocess.run([cuobjdump, "-sass", "-fun", mangled(*key), LIB],
                             capture_output=True, text=True).stdout
        ins = re.findall(r"^\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", txt, flags=re.M)
        assert len(ins) > 500, f"kernel {key} not found in {LIB}"
        out[key] = ins
    return out


@pytest.mark.parametrize("key", FUSED)
def test_fused_kernels_are_warp_uniform_and_spill_free(sass, key):
    ins = sass[key]
    assert not [i for i in ins if "BRA.DIV" in i], "divergence guard in the marching loop"
    assert not [i for i in ins if i.startswith(("STL", "LDL"))], "register spills"
    assert not [i for i in ins if "WARPSYNC" in i and key[3] == 0]


def test_mandatory_math_share_of_the_main_kernel(sass):
    """One marching step = 4 backups = 132 FFMA + 16 FMNMX3; everything else
    (table fetch, ring, shuffles, pointers) must stay below a third of that."""
    ins = sass[(2, 2, 0, 0, 0)]
    stores = [i for i, t in enumerate(ins) if "STG" in t]
    assert len(stores) >= 4
    step = ins[stores[2] + 1:stores[3] + 1]
    ffma = sum(t.startswith("FFMA") or " FFMA" in t for t in step)
    fmn = sum("FMNMX3" in t for t in step)
    assert (ffma, fmn) == (132, 16)
    assert len(step) - ffma - fmn <= 50, f"{len(step)} instructions per step"
    # data movement of the kernel: per-lane cp.async ring, no tensor-core / TMA ops by design
    assert any("LDGSTS" in t for t in ins)
    assert not any(("UTMALDG" in t) or ("UTCMMA" in t) or ("HMMA" in t) for t in ins)
