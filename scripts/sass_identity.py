"""Compare the SASS of every kernel of two builds of librayrs_b200.so, function by function.

    python scripts/sass_identity.py PARENT/rayrs_b200/librayrs_b200.so rayrs_b200/librayrs_b200.so

A function present in the first library must have identical SASS text (instructions and encodings) in the
second.  The anonymous-namespace hash in kernel names depends on the source path and is normalised.  Exit status 1
if any function differs or is missing.
"""
import re
import subprocess
import sys

ANON = re.compile(r"_GLOBAL__N__[0-9a-f]+_")


def functions(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = ANON.sub("_GLOBAL__N__X_", m.group(1))
            res[cur] = []
        elif cur is not None and line.strip().startswith(("/*", ".")):
            res[cur].append(ANON.sub("_GLOBAL__N__X_", line.strip()))
    return res


def main():
    a, b = functions(sys.argv[1]), functions(sys.argv[2])
    same = diff = 0
    for k in sorted(a):
        if k not in b:
            print("MISSING in new:", k)
            diff += 1
        elif a[k] == b[k]:
            same += 1
        else:
            print("DIFFERENT:", k, len(a[k]), len(b[k]))
            diff += 1
    new = sorted(set(b) - set(a))
    print(f"parent functions: {len(a)}, identical: {same}, different/missing: {diff}; new functions: {len(new)}")
    for k in new:
        print("  new:", k)
    sys.exit(1 if diff else 0)


if __name__ == "__main__":
    main()
