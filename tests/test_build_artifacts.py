"""The built library is what DESIGN.md says it is: sm_100a code only, the time sweeps move their data with bulk asynchronous copies
completed on mbarriers (SASS UBLKCP / SYNCS), the candidate ring gathers with cp.async (LDGSTS), the arithmetic is the FP64 pipe and no
tensor-core instruction exists; the hot instantiations keep the register budgets their occupancy was designed for.  Static checks of
the .so with cuobjdump -- no GPU needed; they guard against a build that silently loses the Blackwell path."""
import collections
import os
import re
import shutil
import subprocess

import pytest

from aircraftoptimalcontrol_b200 import build
from tests.util import ROOT

SO = os.path.join(ROOT, "aircraftoptimalcontrol_b200", "libacoc.so")


def _tool(name):
    """A CUDA binary utility from PATH, else the one beside the nvcc that builds the library."""
    return shutil.which(name) or shutil.which(name, path=os.path.dirname(build.NVCC))


CUOBJDUMP, CUFILT = _tool("cuobjdump"), _tool("cu++filt")
pytestmark = pytest.mark.skipif(CUOBJDUMP is None or CUFILT is None or not os.path.exists(SO), reason="cuobjdump, cu++filt or libacoc.so missing")


def _run(*args):
    return subprocess.run([CUOBJDUMP, *args, SO], capture_output=True, text=True, check=True, timeout=300).stdout


def test_only_sm_100a_code():
    elfs = [ln for ln in _run("-lelf").splitlines() if ln.startswith("ELF file")]
    assert elfs and all("sm_100a" in ln for ln in elfs), elfs
    assert "PTX file" not in _run("-lptx")   # no JIT path either: the kernels are compiled for the target, not for a family


def test_register_budgets_of_the_hot_kernels():
    res = _run("-res-usage")
    names = subprocess.run([CUFILT], input="\n".join(re.findall(r"Function (\S+?):", res)), capture_output=True, text=True).stdout.split("\n")
    regs = {}
    for (_, usage), name in zip(re.findall(r"Function (\S+?):\s*\n\s*(.*)", res), names):
        short = re.sub(r"\(.*", "", name.replace("acoc::", "").replace("(bool)", "").replace("(int)", "").replace("void ", ""))
        regs[short] = int(dict(kv.split(":") for kv in usage.split())["REG"])
    # 64-thread CTAs, 7 per SM (the whole 65,536-instance batch in one round) need <= 128 registers; the candidate ring runs 3 CTAs
    # of 320 threads per SM with <= 64; the small-batch pipelines hold 384 threads per SM: <= 168
    assert regs["k_forward_cand0_tma<1, double, float, 1>"] <= 128
    assert regs["k_rollout_write_tma<1, double, float, 1, 1>"] <= 128
    assert regs["k_candidates_list<1, double, 9, 1, 2>"] <= 64
    assert regs["k_backward_cols<1, double, float, 1>"] <= 168 and regs["k_search_fused<1, double, float>"] <= 168
    assert regs["k_backward_tma<1, double, float, 1>"] <= 255


def test_sass_uses_the_blackwell_data_path_and_no_tensor_cores():
    sass = _run("-sass")
    ops = collections.Counter(m.group(1).split(".")[0] for m in re.finditer(r"^\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_.]*)", sass, re.M))
    assert ops["UBLKCP"] > 100 and ops["SYNCS"] > 100      # bulk asynchronous copies + mbarrier waits/arrives of the TMA rings
    assert ops["LDGSTS"] > 0                               # cp.async gathers of the candidate ring
    assert ops["DFMA"] > 1000 and ops["DMUL"] > 1000       # the arithmetic is the FP64 pipe
    for tensor_op in ("HMMA", "IMMA", "DMMA", "QMMA", "UTCMMA", "UTCHMMA"):
        assert ops[tensor_op] == 0, tensor_op              # 6x6 / 2x6 non-dense FP64 contractions: tensor cores unused by design
    # every kernel of the TMA path exists in the binary (a renamed or dropped kernel would make the driver fall back to plain loads)
    for k in ("k_backward_tma", "k_forward_cand0_tma", "k_rollout_write_tma", "k_candidates_list", "k_backward_cols", "k_backward_split",
              "k_search_fused", "k_gradient_tma", "k_deliver", "k_gen_vref"):
        assert re.search(r"Function : \S*%s" % k, sass), k
