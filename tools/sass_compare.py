"""Compare the SASS of two builds of libabfit.so kernel by kernel, ignoring names and addresses.

    python3 tools/sass_compare.py OLD/libabfit.so NEW/libabfit.so

Every kernel of OLD must have a kernel in NEW with an identical instruction body (mangled names may differ, e.g. when
a template gains a defaulted parameter).  Exit status 1 lists the OLD kernels without such a twin."""
import collections
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    fs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name:
                fs[name] = body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line) if name else None
        if m:
            body.append(re.sub(r"\(\*\"[^\"]*\"\*\)", "", m.group(1)).strip())  # symbol names inside operands
    if name:
        fs[name] = body
    return fs


def main(old_path, new_path):
    old, new = kernels(old_path), kernels(new_path)
    bodies = collections.defaultdict(list)
    for n, b in new.items():
        bodies["\n".join(b)].append(n)
    missing = [n for n, b in sorted(old.items()) if "\n".join(b) not in bodies]
    for n in missing:
        print("no identical body in the new build:", n)
    print(f"{len(old)} kernels in the old build, {len(new)} in the new one, {len(missing)} without an identical body")
    return 1 if missing else 0


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
