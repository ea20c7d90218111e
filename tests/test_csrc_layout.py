"""Source layout of the CUDA library: the tcgen05, mbarrier and TMA tensor-copy PTX lives in csrc/tc05.cuh only,
so a fix to a wrapper (a try-wait loop, a descriptor field, a TMA box) is made once and every tensor-core kernel
gets it."""

from __future__ import annotations

import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fast_plaid_b200", "csrc")
HOME = "tc05.cuh"
FAMILIES = ("tcgen05.", "mbarrier.", "cp.async.bulk.tensor")

_TOKEN = re.compile(
    r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"|\'(?:\\.|[^\'\\\n])*\'|[A-Za-z_]\w*|.', re.S)


def asm_strings(text):
    """The PTX template of every asm statement in a C++ source: the string literals before its first colon,
    concatenated.  Comments are skipped by the tokenizer, so prose that names an instruction does not count."""
    toks = [t for t in _TOKEN.findall(text) if not t.startswith(("//", "/*")) and not t.isspace()]
    out = []
    i = 0
    while i < len(toks):
        if toks[i] in ("asm", "__asm__"):
            j = i + 1
            while j < len(toks) and toks[j] in ("volatile", "__volatile__"):
                j += 1
            if j < len(toks) and toks[j] == "(":
                depth, k, ptx, template = 0, j, [], True
                while k < len(toks):
                    if toks[k] == "(":
                        depth += 1
                    elif toks[k] == ")":
                        depth -= 1
                        if depth == 0:
                            break
                    elif toks[k] == ":" and depth == 1:
                        template = False  # operands and clobbers follow
                    elif template and toks[k].startswith('"'):
                        ptx.append(toks[k][1:-1])
                    k += 1
                out.append("".join(ptx))
                i = k
        i += 1
    return out


def test_asm_strings_reads_literals_not_comments():
    src = '''
      // tcgen05.mma in a comment
      /* mbarrier.init in a block comment */
      const char* s = "cp.async.bulk.tensor in a string outside asm";
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm("{\\n" "tcgen05.commit [%0];" "\\n}" :: "r"(bar));
    '''
    assert asm_strings(src) == ["fence.proxy.async.shared::cta;", "{\\ntcgen05.commit [%0];\\n}"]


def test_tensor_core_ptx_lives_in_tc05_only():
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    home = "".join(asm_strings(open(os.path.join(CSRC, HOME)).read()))
    assert all(f in home for f in FAMILIES), "the scanner found no tcgen05 / mbarrier / TMA PTX in tc05.cuh"
    offenders = []
    for name in sources:
        if name == HOME:
            continue
        for ptx in asm_strings(open(os.path.join(CSRC, name)).read()):
            offenders += [(name, f, ptx) for f in FAMILIES if f in ptx]
    assert not offenders, f"tcgen05 / mbarrier / TMA PTX outside {HOME}: {offenders}"
