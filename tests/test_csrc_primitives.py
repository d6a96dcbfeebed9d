"""Every inline-PTX instruction string of the CUDA sources is written once: the kernels call the wrappers in
common.cuh, tma.cuh and tc.cuh instead of carrying private copies that drift apart."""
import re
from collections import defaultdict
from pathlib import Path

CSRC = Path(__file__).resolve().parents[1] / "spotv2net_b200" / "csrc"
ASM = re.compile(r'\basm\s*(?:volatile\s*)?\(\s*((?:"(?:[^"\\]|\\.)*"\s*)+)')
LITERAL = re.compile(r'"((?:[^"\\]|\\.)*)"')

# instruction string -> (places it may appear, why)
ALLOWED = {
    "ld.shared.f32 %0, [%1];": (2, "lds_f32 (plain asm, free to be hoisted) and lds_f32_v (asm volatile, issued where written)"),
}


def asm_strings():
    where = defaultdict(list)
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh"))):
        text = f.read_text()
        for m in ASM.finditer(text):
            s = " ".join("".join(LITERAL.findall(m.group(1))).split())
            where[s].append(f"{f.name}:{text.count(chr(10), 0, m.start()) + 1}")
    return where


def test_sources_have_inline_asm():
    where = asm_strings()
    assert len(where) > 40
    assert "mbarrier.arrive.shared::cta.b64 _, [%0];" in where


def test_each_asm_string_written_once():
    repeated = {s: w for s, w in asm_strings().items() if len(w) > ALLOWED.get(s, (1, ""))[0]}
    assert not repeated, "inline asm written in more than one place (call the shared wrapper instead):\n" + "\n".join(
        f"  {s!r}: {', '.join(w)}" for s, w in repeated.items())


def test_allow_list_is_current():
    where = asm_strings()
    assert all(len(where.get(s, [])) == n for s, (n, _) in ALLOWED.items())
