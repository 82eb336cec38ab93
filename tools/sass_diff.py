"""Kernel-by-kernel SASS comparison of two builds of libvrm_b200.so.

    python tools/sass_diff.py OLD.so NEW.so

Prints, for every kernel of OLD, whether NEW has it with identical instructions.  Instruction addresses, the fatbin headers between
cubins and the per-translation-unit hash of anonymous-namespace names are ignored; everything else of `cuobjdump -sass` must match.
Exit status 1 when a kernel of OLD changed or is missing in NEW.  Used to show that a change adds kernels without touching any
existing one: build the parent commit's library in a scratch checkout and compare it with the branch build.
"""
import argparse
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def kernels(so):
    out = subprocess.run([CUOBJDUMP, "-sass", so], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
        elif name and "/*" in line:  # instruction lines only: "/*0040*/ OPCODE ... ;  /* 0x... */" and the encoding continuation lines
            body.append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip())
    if name:
        funcs[name] = body
    # anonymous namespace: _ZN<len>_GLOBAL__N__<hash>_<n>_<file>_cu_<hash><len><name> -> ANON(<file>)<name>
    norm = lambda n: re.sub(r"_ZN\d+_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]{8}\d+", r"ANON(\1)", n)  # noqa: E731
    return {norm(k): v for k, v in funcs.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("old")
    ap.add_argument("new")
    a = ap.parse_args()
    old, new = kernels(a.old), kernels(a.new)
    same = [k for k in old if k in new and old[k] == new[k]]
    changed = [k for k in old if k in new and old[k] != new[k]]
    missing = [k for k in old if k not in new]
    added = [k for k in new if k not in old]
    print(f"{len(old)} kernels in {a.old}, {len(new)} in {a.new}: {len(same)} identical, {len(changed)} changed, {len(missing)} missing, "
          f"{len(added)} new")
    for k in changed:
        print("  changed:", k)
    for k in missing:
        print("  missing:", k)
    for k in added:
        print("  new:    ", k)
    return 1 if changed or missing else 0


if __name__ == "__main__":
    sys.exit(main())
