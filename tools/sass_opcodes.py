"""Per-kernel digest of the SASS opcode stream of libmipnerf_b200.so (`cuobjdump -sass`): instruction count and a
sha256 of the opcode sequence (mnemonic with its modifiers, predicates and operands dropped), plus registers from
`cuobjdump --dump-resource-usage`.  Operands are left out on purpose: a kernel parameter struct that grows moves the
constant-bank offsets of the loads without changing the code.

    python tools/sass_opcodes.py [LIB] [--match mlp_level_kernel] > digest.json
"""
from __future__ import annotations

import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
from typing import Dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "mipnerf_pl_b200", "libmipnerf_b200.so")
_INSN = re.compile(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)")


def cuobjdump() -> str:
    for cand in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"),
                 shutil.which("cuobjdump")):
        if cand and os.path.exists(cand):
            return cand
    raise FileNotFoundError("cuobjdump not found")


def _key(mangled: str, match: str) -> str:
    """The mangled name from `match` on: drops the anonymous-namespace prefix, whose hash changes with the source."""
    return mangled[mangled.index(match):]


def digest(lib: str = DEFAULT_LIB, match: str = "mlp_level_kernel") -> Dict[str, dict]:
    """{mangled kernel name from `match` on: {'insns', 'sha256', 'regs'}} for the kernels whose name contains `match`."""
    tool = cuobjdump()
    sass = subprocess.run([tool, "-sass", lib], capture_output=True, text=True, check=True).stdout
    out: Dict[str, dict] = {}
    name, ops = None, []

    def flush():
        if name is not None and match in name:
            out[_key(name, match)] = {"insns": len(ops), "sha256": hashlib.sha256("\n".join(ops).encode()).hexdigest()}

    for line in sass.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            flush()
            name, ops = m.group(1), []
            continue
        m = _INSN.search(line)
        if m and name is not None:
            ops.append(m.group(1))
    flush()
    res = subprocess.run([tool, "--dump-resource-usage", lib], capture_output=True, text=True, check=True).stdout
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+)", res):
        if match in m.group(1) and _key(m.group(1), match) in out:
            out[_key(m.group(1), match)]["regs"] = int(m.group(2))
    return out


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    match = sys.argv[sys.argv.index("--match") + 1] if "--match" in sys.argv else "mlp_level_kernel"
    if "--match" in sys.argv:
        args.remove(match)
    json.dump(digest(args[0] if args else DEFAULT_LIB, match), sys.stdout, indent=1, sort_keys=True)
    print()
