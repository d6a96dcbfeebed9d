"""Compare the machine code of two builds of libspotv2_gat.so, function by function.

    python tools/sass_diff.py OLD NEW

OLD and NEW are each a package directory (libspotv2_gat.so and its _build/), a _build/ directory (the .o files are
read) or a libspotv2_gat.so.  The SASS comes from `cuobjdump -sass`; before the comparison only code addresses, the
encoding comments and the targets of relative BRA / CALL are masked.  Names in anonymous namespaces carry an id that
nvcc draws per compilation (`_GLOBAL__N__<id>_13_attn_fwd_cu_...`); it is masked so that the two builds' functions pair
up.  The `-Xptxas -v` lines of the _build/*.log files (registers, barriers, shared memory, stack, spills) are compared
too.  Prints every function that differs and exits 1 if any does, 0 if none.
"""
from __future__ import annotations

import re
import shutil
import subprocess
import sys
from collections import defaultdict
from pathlib import Path

FUNC = re.compile(r"^\s*Function : (\S+)")
INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*(?:/\*\s*0x[0-9a-f]+\s*\*/)?\s*$")
ENCODING_ONLY = re.compile(r"^\s*/\*\s*0x[0-9a-f]+\s*\*/\s*$")
REL_TARGET = re.compile(r"^((?:@!?U?P\w+\s+)?(?:BRA|CALL\.REL)\S*\s.*?)0x[0-9a-f]+(\s*)$")
# ptxas -v lines that describe a function (compile times and the like are left out)
PTXAS_FUNC = re.compile(r"(?:Compiling entry function|Function properties for) '?([^' ]+)'?")
PTXAS_KEEP = re.compile(r"registers|stack|spill|smem|cmem|gmem|barriers")
COMPILATION_ID = re.compile(r"(_GLOBAL__N__|_INTERNAL_)[0-9a-f]{8}_")


def _unid(s: str) -> str:
    return COMPILATION_ID.sub(r"\1_", s)


def _cuobjdump() -> str:
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand and Path(cand).exists():
            return cand
    sys.exit("cuobjdump not found")


def _inputs(path: Path) -> tuple[list[Path], list[Path]]:
    """(binaries to disassemble, ptxas logs) of one build."""
    if path.is_file():
        return [path], sorted((path.parent / "_build").glob("*.log"))
    if (path / "libspotv2_gat.so").exists():
        return [path / "libspotv2_gat.so"], sorted((path / "_build").glob("*.log"))
    objs = sorted(path.glob("*.o"))
    if not objs:
        sys.exit(f"{path}: neither libspotv2_gat.so nor .o files")
    return objs, sorted(path.glob("*.log"))


def sass_by_function(binaries: list[Path]) -> dict[str, list[str]]:
    out: dict[str, list[str]] = {}
    for b in binaries:
        res = subprocess.run([_cuobjdump(), "-sass", str(b)], capture_output=True, text=True)
        if res.returncode != 0:
            sys.exit(f"cuobjdump -sass {b} failed:\n{res.stderr}")
        name, body = None, []
        for line in _unid(res.stdout).splitlines() + ["\t\tFunction : <end>"]:
            m = FUNC.match(line)
            if m:
                if name is not None:
                    key, n = name, 1
                    while key in out:                  # same name in two objects: keep both, in order
                        n += 1
                        key = f"{name}#{n}"
                    out[key] = body
                name, body = m.group(1), []
                continue
            if name is None or ENCODING_ONLY.match(line):
                continue
            m = INSN.match(line)
            if m:
                insn = " ".join(m.group(1).split())
                body.append(REL_TARGET.sub(r"\1<target>\2", insn))
            elif line.strip() and not line.strip().startswith(("code for", ".target", "Fatbin", "===", "arch =", "code version",
                                                                "host =", "compile_size", "identifier", "compressed")):
                body.append(" ".join(line.split()))
        if name is not None and name != "<end>":
            out[name] = body
    out.pop("<end>", None)
    return out


def ptxas_by_function(logs: list[Path]) -> dict[str, list[str]]:
    out: dict[str, list[str]] = defaultdict(list)
    for log in logs:
        current = f"<{log.name}>"
        for line in _unid(log.read_text()).splitlines():
            m = PTXAS_FUNC.search(line)
            if m:
                current = m.group(1)
            elif PTXAS_KEEP.search(line) and "Compile time" not in line:
                out[current].append(" ".join(line.replace("ptxas info    :", "").split()))
    return out


def main(argv: list[str]) -> int:
    if len(argv) != 3:
        sys.exit(__doc__)
    old, new = Path(argv[1]), Path(argv[2])
    (ob, ol), (nb, nl) = _inputs(old), _inputs(new)
    differ = []
    for what, a, b in (("sass", sass_by_function(ob), sass_by_function(nb)),
                       ("ptxas", ptxas_by_function(ol), ptxas_by_function(nl))):
        for name in sorted(set(a) | set(b)):
            if name not in a or name not in b:
                differ.append(f"{what}: {name}: only in {'new' if name in b else 'old'}")
            elif a[name] != b[name]:
                i = next((k for k, (x, y) in enumerate(zip(a[name], b[name])) if x != y), min(len(a[name]), len(b[name])))
                first = lambda s: s[i] if i < len(s) else "<end>"
                differ.append(f"{what}: {name}: {len(a[name])} -> {len(b[name])} lines, first difference at line {i}:\n"
                              f"    old: {first(a[name])}\n    new: {first(b[name])}")
        print(f"{what}: {len(a)} functions in old, {len(b)} in new")
    for d in differ:
        print(d)
    print(f"{len(differ)} differing function(s)")
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
