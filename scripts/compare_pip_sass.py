"""Compare the SASS of the point-in-polygon kernels of two builds (no GPU needed).

    python scripts/compare_pip_sass.py OLD NEW [--out FILE]

OLD and NEW are libsegger_b200.so files or sgb_pip.cu objects.  Every instantiation of ``pip_polygon_kernel`` and
``polygon_props_kernel`` in OLD must have the same instructions in NEW.  A template flag added with a default of
``false`` (``BUF``, then ``MULTI``) is matched to the instantiation with that flag false; addresses, encodings and the
per-build hash of the anonymous namespace are ignored.  Prints one line per kernel and exits non-zero on a difference.
"""
from __future__ import annotations

import argparse
import re
import subprocess
import sys

KERNELS = ("pip_polygon_kernel", "polygon_props_kernel")


def _sass(path: str) -> dict[str, list[str]]:
    out = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        if name is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*(/\*.*\*/)?\s*$", line)
        if m and m.group(1):
            funcs[name].append(re.sub(r"_GLOBAL__N__\w+?_cu_\w+?(?=\d)", "_ANON_", m.group(1)))
    return funcs


def _key(mangled: str) -> str | None:
    for k in KERNELS:
        i = mangled.find(f"{len(k)}{k}")
        if i < 0:
            continue
        rest = mangled[i + len(f"{len(k)}{k}"):]
        flags = re.match(r"I((?:Lb[01]E)+)E", rest)
        bits = re.findall(r"Lb([01])E", flags.group(1)) if flags else []
        while bits and bits[-1] == "0" and len(bits) > 2:        # a trailing flag added later with default false
            bits.pop()
        return k + (f"<{','.join(bits)}>" if bits else "")
    return None


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out")
    a = ap.parse_args()
    old = {k: v for n, v in _sass(a.old).items() if (k := _key(n))}
    new = {k: v for n, v in _sass(a.new).items() if (k := _key(n))}
    lines, bad = [], 0
    for k in sorted(old):
        same = new.get(k) == old[k]
        bad += not same
        lines.append(f"{k}: {len(old[k])} instructions, {'identical' if same else 'DIFFERENT'}")
    extra = sorted(set(new) - set(old))
    lines.append(f"new instantiations only in NEW: {', '.join(extra) if extra else 'none'}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 1 if bad or not old else 0


if __name__ == "__main__":
    sys.exit(main())
