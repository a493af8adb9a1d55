#!/usr/bin/env python
"""Compare the SASS of every kernel in two builds of libcolosseum_b200.so, function by function (dev helper).

usage: python tools/sass_compare.py OLD.so NEW.so [--rename=OLD_NAME=NEW_NAME ...]

Each kernel's instructions are compared with the instruction addresses stripped, so a kernel that only moved inside
the binary compares equal.  --rename pairs a kernel whose mangled name changed (a new template parameter, appended
parameters) with its new name.  Prints SAME / DIFF per kernel of OLD, MISSING for kernels gone, NEW for added ones;
exits 1 if any kernel of OLD differs or is missing.
"""
import re
import subprocess
import sys


def kernels(so):
    text = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name:
            out[name].append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip())
    return out


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--rename")]
    ren = dict(a[len("--rename="):].split("=", 1) for a in sys.argv[1:] if a.startswith("--rename="))
    if len(args) < 2:
        sys.exit(__doc__)
    old, new = kernels(args[0]), kernels(args[1])
    bad = 0
    for k, body in old.items():
        k2 = ren.get(k, k)
        if k2 not in new:
            print("MISSING", k)
            bad += 1
        else:
            same = new[k2] == body
            print("SAME" if same else "DIFF", k, "" if k2 == k else "-> " + k2)
            bad += not same
    for k in sorted(set(new) - {ren.get(k, k) for k in old}):
        print("NEW", k)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
