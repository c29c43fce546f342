"""tools/sass_diff.py OLD.so NEW.so -- compare the SASS of every kernel of two builds of libf110_b200.so, function by function.

Names are matched with the anonymous-namespace hash removed (it depends on the build directory).  Prints one line per
function of OLD whose instructions differ in NEW (or that NEW lacks), then a summary line; the functions only NEW has
are listed by name.  Exit status 1 when any function of OLD differs.
"""
import os
import re
import shutil
import subprocess
import sys


def functions(so):
    tool = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.check_output([tool, "-sass", so]).decode()
    fns, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function\s*:\s*(\S+)", line)
        if m:
            name = re.sub(r"_GLOBAL__N__\w+?_cu_[0-9a-f]+", "ANON", m.group(1))
            fns[name] = []
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?)\s*;", line)
        if m and name:
            fns[name].append(m.group(2).strip())
    return fns


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    same = 0
    for k in sorted(old):
        if k not in new:
            print("missing in NEW:", k)
        elif old[k] != new[k]:
            moved = sum(x != y for x, y in zip(old[k], new[k])) + abs(len(old[k]) - len(new[k]))
            print("differs: %s (%d vs %d instructions, %d lines differ)" % (k, len(old[k]), len(new[k]), moved))
        else:
            same += 1
    print("OLD functions: %d, identical in NEW: %d, different or missing: %d; only in NEW: %d"
          % (len(old), same, len(old) - same, len(set(new) - set(old))))
    for k in sorted(set(new) - set(old)):
        print("  new:", k)
    return 0 if same == len(old) else 1


if __name__ == "__main__":
    sys.exit(main())
