"""Is the SASS of every k_history instantiation of a git revision unchanged in the working tree?
Compiles neutral_b200/csrc/history.cu of both for sm_100a with the library's own nvcc flags
(nvcc -cubin, no GPU needed), disassembles them with cuobjdump -sass, and compares the
instantiations that exist in both, keyed by their leading template arguments (F/T for each
bool; an instantiation of the tree with one more trailing `false` argument is the same variant).
Symbol names and instruction addresses are stripped, so a changed kernel signature alone does
not count; encodings, constant-bank offsets and branch targets do. Prints ptxas's registers,
spills and shared memory for the tree's instantiations.

    python tools/sass_identity.py HEAD          # exit status 1 if any shared variant differs
"""
from __future__ import annotations

import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from neutral_b200.build import NVCC_FLAGS, find_nvcc  # noqa: E402


def sass_by_variant(csrc: str, out: str) -> dict:
    cubin = out + ".cubin"
    res = subprocess.run([find_nvcc()] + NVCC_FLAGS + ["-cubin", os.path.join(csrc, "history.cu"),
                                                       "-o", cubin],
                         capture_output=True, text=True, check=True)
    ptxas = res.stdout + res.stderr
    dump = subprocess.run([os.path.join(os.path.dirname(find_nvcc()), "cuobjdump"), "-sass",
                           cubin], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\t\tFunction : (\S+)\n", dump)
    variants = {}
    for name, body in zip(parts[1::2], parts[2::2]):
        m = re.search(r"k_historyI((?:Lb[01]E)+)", name)
        if not m:
            continue
        key = "".join("T" if b == "1" else "F" for b in re.findall(r"Lb([01])E", m.group(1)))
        body = re.sub(r"_Z\w+", "<sym>", body)
        body = re.sub(r"/\*[0-9a-f]{4,}\*/", "", body)
        variants[key] = [ln.strip() for ln in body.splitlines() if ln.strip()]
    return variants, ptxas


def main() -> int:
    rev = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
    with tempfile.TemporaryDirectory() as tmp:
        old_tree = os.path.join(tmp, "old")
        os.makedirs(old_tree)
        archive = subprocess.run(["git", "-C", ROOT, "archive", rev, "neutral_b200/csrc",
                                  "include"], capture_output=True, check=True).stdout
        subprocess.run(["tar", "-x", "-C", old_tree], input=archive, check=True)
        old, _ = sass_by_variant(os.path.join(old_tree, "neutral_b200", "csrc"),
                                 os.path.join(tmp, "old"))
        new, ptxas = sass_by_variant(os.path.join(ROOT, "neutral_b200", "csrc"),
                                     os.path.join(tmp, "new"))
    for line in ptxas.splitlines():
        if "k_history" in line and "Compiling entry" in line:
            print(line.split("'")[1])
        elif "registers" in line or "spill" in line:
            print("   ", line.strip())
    differs = 0
    for key, body in sorted(old.items()):
        match = next((k for k in new if k == key or (k.startswith(key) and
                                                       set(k[len(key):]) == {"F"})), None)
        if match is None:
            print(f"{key}: gone from the tree")
            differs += 1
        elif new[match] == body:
            print(f"{key}: identical to {rev} ({len(body)} lines)")
        else:
            print(f"{key}: DIFFERS from {rev}")
            differs += 1
    return 1 if differs else 0


if __name__ == "__main__":
    sys.exit(main())
