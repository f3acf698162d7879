"""Compare the machine code of every kernel of two builds, function by function, with control words.

    python profiles/tools/sass_diff.py <old build dir> <new build dir>

Each directory holds the object files tinympc-matlab_b200/build.py writes (tinympc-matlab_b200/build/*.o).  For every kernel of
the old build the script compares `cuobjdump -sass` of the same symbol in the new build, instructions and the /* 0x... */
encoding words (which carry the control bits: stall counts, barriers, reuse flags).  It prints one line per object file and a
summary; the exit code is 1 when an old kernel changed or disappeared.
"""
import re
import subprocess
import sys
from pathlib import Path

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def functions(obj: Path) -> dict:
    txt = subprocess.run([CUOBJDUMP, "-sass", str(obj)], capture_output=True, text=True).stdout
    out, name, body = {}, None, []
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:   # kernels in an anonymous namespace carry a hash of the translation unit's path: drop it
            if name:
                out[name] = "\n".join(body)
            name, body = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1)), []
        elif name is not None and ("/*" in line):
            body.append(re.sub(r"\s+", " ", line.strip()))
    if name:
        out[name] = "\n".join(body)
    return out


def main(old_dir: str, new_dir: str) -> int:
    old, new = Path(old_dir), Path(new_dir)
    same = changed = gone = added = 0
    for o in sorted(old.glob("*.o")):
        fo = functions(o)
        n = new / o.name
        fn = functions(n) if n.exists() else {}
        s = sum(1 for k in fo if fn.get(k) == fo[k])
        c = [k for k in fo if k in fn and fn[k] != fo[k]]
        g = [k for k in fo if k not in fn]
        a = [k for k in fn if k not in fo]
        same += s; changed += len(c); gone += len(g); added += len(a)
        if fo or fn:
            print(f"{o.name}: {s} identical, {len(c)} changed, {len(g)} missing, {len(a)} new" + "".join(f"\n  changed {k}" for k in c)
                  + "".join(f"\n  missing {k}" for k in g) + "".join(f"\n  new {k}" for k in a))
    print(f"TOTAL: {same} kernels identical, {changed} changed, {gone} missing, {added} new")
    return 1 if changed or gone else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
