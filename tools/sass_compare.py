"""Compare two builds of a CUDA library kernel by kernel: same name, same SASS (instruction words and encodings,
with the address column dropped).  Needs cuobjdump, no GPU.

    python tools/sass_compare.py OLD.so NEW.so     # exit status 1 if a kernel of OLD is missing or differs in NEW
"""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def kernels(path):
    out = subprocess.run([CUOBJDUMP, "-sass", path], capture_output=True, text=True, check=True).stdout
    ks, cur, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m or line.strip().startswith("Fatbin"):
            if cur:
                ks[cur] = body
            cur, body = (m.group(1) if m else None), []
        elif cur is not None and line.strip():
            body.append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip())
    if cur:
        ks[cur] = body
    return ks


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    missing = [k for k in a if k not in b]
    differ = [k for k in a if k in b and a[k] != b[k]]
    added = [k for k in b if k not in a]
    print("%d kernels in %s, %d in %s: %d identical, %d differ, %d missing, %d added"
          % (len(a), sys.argv[1], len(b), sys.argv[2], len(a) - len(differ) - len(missing), len(differ), len(missing), len(added)))
    for name, ks in (("differ", differ), ("missing", missing), ("added", added)):
        for k in ks:
            print("  %s: %s" % (name, k))
    return 1 if differ or missing else 0


if __name__ == "__main__":
    sys.exit(main())
