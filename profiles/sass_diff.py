"""Compare the SASS of two builds of nodal_b200/csrc, per object file (= per cubin) and per function.

    python profiles/sass_diff.py <old_build_dir> <new_build_dir> [--rename REGEX=REPL ...]

Each directory holds the object files the Makefile writes (nodal_b200/csrc/build/*.o).  Every
`Function :` block of `cuobjdump -sass` is keyed by (object file, demangled name); the instruction
text is compared with the addresses and encodings removed.  Prints the functions that exist only in
the old build, only in the new one, and those whose instructions differ.  --rename rewrites demangled
names of the old build before matching (for a template parameter that became a constant).
"""
import argparse
import glob
import os
import re
import subprocess
import sys

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def functions(obj):
    sass = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", obj], check=True,
                          capture_output=True, text=True).stdout
    out, name, body = {}, None, []
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*/\* 0x[0-9a-f]+ \*/\s*$", line)
        if m:
            body.append(m.group(1))
    if name:
        out[name] = body
    if not out:
        return {}
    names = list(out)
    dem = subprocess.run([os.path.join(CUDA, "bin", "cu++filt")], input="\n".join(names), check=True,
                         capture_output=True, text=True).stdout.splitlines()
    return {d: out[n] for n, d in zip(names, dem)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--rename", action="append", default=[])
    a = ap.parse_args()
    renames = [r.split("=", 1) for r in a.rename]
    only_old, only_new, differ, same = [], [], [], 0
    objs = sorted({os.path.basename(p) for d in (a.old, a.new) for p in glob.glob(os.path.join(d, "*.o"))})
    for o in objs:
        fo = functions(os.path.join(a.old, o)) if os.path.exists(os.path.join(a.old, o)) else {}
        fn = functions(os.path.join(a.new, o)) if os.path.exists(os.path.join(a.new, o)) else {}
        for pat, repl in renames:
            fo = {re.sub(pat, repl, k): v for k, v in fo.items()}
        for k in sorted(set(fo) | set(fn)):
            if k not in fn:
                only_old.append(f"{o}: {k}")
            elif k not in fo:
                only_new.append(f"{o}: {k}")
            elif fo[k] != fn[k]:
                differ.append(f"{o}: {k}")
            else:
                same += 1
    print(f"identical functions: {same}")
    for title, items in (("only in old", only_old), ("only in new", only_new), ("instructions differ", differ)):
        print(f"{title}: {len(items)}")
        for it in items:
            print("  " + it)
    return 1 if (only_new or differ) else 0


if __name__ == "__main__":
    sys.exit(main())
