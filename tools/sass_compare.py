"""Kernel-by-kernel SASS comparison of two builds of libgpk.so (cuobjdump -sass; no GPU needed).

    python tools/sass_compare.py OLD/libgpk.so NEW/libgpk.so

Prints the kernels only one build has and the kernels whose instructions differ; exits 1 if any differ.  Anonymous-namespace
hashes (which change with every compilation) and instruction addresses are stripped before the comparison, so a change that
only adds host code or a new translation unit reports every existing kernel as identical."""
import re
import subprocess
import sys

_ANON = re.compile(r"_GLOBAL__N__[0-9a-f]+_")


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    ks, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m or "Fatbin elf code" in line:
            if name:
                ks[name] = "\n".join(body)
            name, body = (_ANON.sub("_GLOBAL__N__", m.group(1)) if m else None), []
        elif name is not None and re.search(r"/\*[0-9a-f]{4}\*/", line):
            body.append(_ANON.sub("_GLOBAL__N__", re.sub(r"/\*[0-9a-f]{4}\*/", "", line)).strip())
    if name:
        ks[name] = "\n".join(body)
    return ks


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    changed = sorted(k for k in old.keys() & new.keys() if old[k] != new[k])
    for k in sorted(old.keys() - new.keys()):
        print("only in old:", k)
    for k in sorted(new.keys() - old.keys()):
        print("only in new:", k)
    for k in changed:
        print("changed:", k)
    print(f"{len(old.keys() & new.keys()) - len(changed)} of {len(old)} kernels identical")
    sys.exit(1 if changed or old.keys() - new.keys() else 0)


if __name__ == "__main__":
    main()
