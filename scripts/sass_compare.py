"""Compares the SASS of every kernel present in two builds (cuobjdump -sass output of libmeao.so or of single cubins).

    python scripts/sass_compare.py OLD.sass NEW.sass

A kernel counts as unchanged when its instruction text is byte-identical.  The per-file hash that nvcc puts into the names
of anonymous-namespace symbols is normalised away (it follows the file's content, not the kernel's).  Kernels that exist
only in NEW are listed with whether they contain UTMALDG.3D (3-D TMA loads).  Exit code 1 if a kernel of OLD changed or
disappeared.
"""
from __future__ import annotations

import re
import sys

_ANON = re.compile(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+")


def kernels(path: str) -> dict[str, str]:
    out: dict[str, list[str]] = {}
    cur = None
    for line in open(path, encoding="utf-8", errors="replace"):
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = _ANON.sub(r"anon_\1", m.group(1))
            out[cur] = []
            continue
        if cur is not None and line.strip().startswith("/*") and "*/" in line:
            out[cur].append(_ANON.sub(r"anon_\1", line.strip()))
    return {k: "\n".join(v) for k, v in out.items()}


def main(old_path: str, new_path: str) -> int:
    old, new = kernels(old_path), kernels(new_path)
    bad = 0
    for name in sorted(old):
        if name not in new:
            print(f"MISSING  {name}")
            bad += 1
        elif old[name] != new[name]:
            print(f"CHANGED  {name}")
            bad += 1
        else:
            print(f"same     {name}")
    for name in sorted(set(new) - set(old)):
        print(f"new      {name}  UTMALDG.3D={'yes' if 'UTMALDG.3D' in new[name] else 'no'}")
    print(f"{len(old) - bad} of {len(old)} existing kernels identical; {len(set(new) - set(old))} new")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
