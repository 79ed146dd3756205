"""Compare two builds of a CUDA library kernel by kernel: same name, same SASS (instruction words and encodings,
with the address column dropped).  Needs cuobjdump and cu++filt, no GPU.

    python tools/sass_compare.py OLD.so NEW.so [--rename PATTERN=REPLACEMENT ...]

Kernels are matched by demangled name without the parameter list, an empty template pack counting as absent
(`k<(int)4, >` and `k<>` match `k<(int)4>` and `k`).  --rename applies a regular expression to the old build's names
before matching, in the order given, e.g. to compare a kernel renamed into a template instantiation:

    --rename '_bnd<(.*)>$=<\\1, fe::GateCount>' --rename '_bnd$=<fe::GateCount>'

Exit status 1 if a kernel of OLD is missing or differs in NEW.
"""
import argparse
import os
import re
import subprocess
import sys

CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def kernels(path):
    out = subprocess.run([os.path.join(CUDA_BIN, "cuobjdump"), "-sass", path], capture_output=True, text=True, check=True).stdout
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


def by_name(ks, renames=()):
    """{demangled name without parameters, empty packs dropped, renamed: SASS}"""
    mangled = list(ks)
    out = subprocess.run([os.path.join(CUDA_BIN, "cu++filt"), "-p"], input="\n".join(mangled) + "\n", capture_output=True,
                         text=True, check=True).stdout.splitlines()
    assert len(out) == len(mangled)
    named = {}
    for m, name in zip(mangled, out):
        name = name.strip().replace(", >", ">").replace("<>", "")
        for pat, rep in renames:
            name = re.sub(pat, rep, name)
        if name in named:
            sys.exit("two kernels are both named %s" % name)
        named[name] = ks[m]
    return named


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--rename", action="append", default=[], metavar="PATTERN=REPLACEMENT",
                    help="regular expression substitution applied to the old build's kernel names (repeatable)")
    args = ap.parse_args()
    renames = []
    for r in args.rename:
        pat, sep, rep = r.partition("=")
        if not sep:
            ap.error("--rename takes PATTERN=REPLACEMENT: %r" % r)
        renames.append((pat, rep))
    a, b = by_name(kernels(args.old), renames), by_name(kernels(args.new))
    missing = [k for k in a if k not in b]
    differ = [k for k in a if k in b and a[k] != b[k]]
    added = [k for k in b if k not in a]
    print("%d kernels in %s, %d in %s: %d identical, %d differ, %d missing, %d added"
          % (len(a), args.old, len(b), args.new, len(a) - len(differ) - len(missing), len(differ), len(missing), len(added)))
    for name, ks in (("differ", differ), ("missing", missing), ("added", added)):
        for k in ks:
            print("  %s: %s" % (name, k))
    return 1 if differ or missing else 0


if __name__ == "__main__":
    sys.exit(main())
