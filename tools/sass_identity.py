"""Compare the SASS of two builds of the library, kernel by kernel.

    python tools/sass_identity.py OLD_BUILD_DIR NEW_BUILD_DIR

Each directory holds the .o files of `python -m torch_admm_deconv_b200.build` (torch_admm_deconv_b200/build/).  Every
kernel of OLD must appear in NEW with identical instructions; addresses, encodings and the `Function :` names are
normalised away, and the names of kernels that became templates on the real type are mapped back (`k_rows<2, float>` ->
`k_rows<2>`, `RowArgsT<float>` -> `RowArgs`, ...).  Kernels only NEW has are listed.  Exit status 1 if any OLD kernel
differs or is missing.  Used to show that templating the generic engine on the element type left the float32 library
bit-identical."""
import os
import re
import subprocess
import sys


def cuobjdump():
    for c in (os.environ.get("CUOBJDUMP"), "/usr/local/cuda/bin/cuobjdump", "cuobjdump"):
        if c and (os.path.sep not in c or os.path.exists(c)):
            return c
    return "cuobjdump"


def functions(obj):
    out = subprocess.run([cuobjdump(), "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
            continue
        if cur is None:
            continue
        line = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)           # instruction addresses
        line = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", line).strip()   # encodings
        if line:
            res[cur].append(line)
    return res


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, r))


def key(d):
    d = re.sub(r"^void ", "", d)
    d = d.replace("admm::cplx_of<float>::type", "float2")
    d = d.replace("admm::RowArgsT<float>", "admm::RowArgs").replace("admm::ColArgsT<float>", "admm::ColArgs")
    d = re.sub(r"k_(rows|cols)<(\d+), float>", r"k_\1<\2>", d)
    d = re.sub(r"<(true|false), float>\(", r"<\1>(", d)
    d = re.sub(r"<float2?>\(", "(", d)
    return d


def main():
    old, new = sys.argv[1], sys.argv[2]
    total = same = 0
    bad, added = [], []
    for f in sorted(os.listdir(old)):
        if not f.endswith(".o"):
            continue
        fo = functions(os.path.join(old, f))
        fn = functions(os.path.join(new, f)) if os.path.exists(os.path.join(new, f)) else {}
        do, dn = demangle(list(fo)), demangle(list(fn))
        ko, kn = {key(do[n]): n for n in fo}, {key(dn[n]): n for n in fn}
        for k, n in ko.items():
            total += 1
            if k not in kn:
                bad.append((f, k, "missing"))
            elif fo[n] == fn[kn[k]]:
                same += 1
            else:
                bad.append((f, k, "differs"))
        added += [(f, k) for k in kn if k not in ko]
    print("kernels in %s: %d, SASS-identical in %s: %d" % (old, total, new, same))
    for b in bad:
        print("DIFFERS" if b[2] == "differs" else "MISSING", b[0], b[1])
    for a in added:
        print("NEW", a[0], a[1])
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
