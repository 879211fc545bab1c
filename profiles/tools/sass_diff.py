"""Compares the SASS of two libba_cuda.so builds kernel by kernel.

usage: sass_diff.py PARENT.so BRANCH.so

Each kernel is the instruction text of `cuobjdump -sass`: encodings are dropped and the hash of the anonymous
namespace is masked, so two builds of the same source compare equal.  Kernels are matched by demangled name
without the parameter list.  RENAMES maps a parent kernel that a change merged into another to the kernel that
replaces it; it is applied only when the parent name is gone from the branch build.

Exit status 0 when every parent kernel outside RENAMES is in the branch build with the same instructions.
"""
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"

# r06 (one linearisation driver for tiles and strips): the strip copies of the per-camera kernels became
# instantiations of their tile counterparts, which gained a template parameter for where diag F^T F sits.
RENAMES = {
    "ba::k_jacobi_scale<3, 9>": "ba::k_jacobi_scale<3, 9, -1>",
    "ba::k_jacobi_scale<6, 27>": "ba::k_jacobi_scale<6, 27, -1>",
    "ba::k_jacobi_scale<6, 33>": "ba::k_jacobi_scale<6, 33, -1>",
    "ba::k_sa_jacobi_scale": "ba::k_jacobi_scale<6, 39, 33>",
    "ba::k_fa_scale_cams": "ba::k_fa_scale_cams<33>",
    "ba::k_sa_scale_cams": "ba::k_fa_scale_cams<39>",
    "ba::k_diag_rhs_bsr": "ba::k_diag_rhs_bsr<-1>",
    "ba::k_diag_rhs_dense": "ba::k_diag_rhs_dense<-1>",
    "ba::k_sa_diag_rhs_bsr": "ba::k_diag_rhs_bsr<33>",
    "ba::k_sa_diag_rhs_dense": "ba::k_diag_rhs_dense<33>",
}

ANON = re.compile(r"_GLOBAL__N__[0-9A-Za-z_]+?_[0-9a-f]{8}")


def short_name(demangled):
    """'void ba::k<6, 33>(long, double*)' -> 'ba::k<6, 33>'"""
    depth = 0
    for i, c in enumerate(demangled):
        if c == "<":
            depth += 1
        elif c == ">":
            depth -= 1
        elif c == "(" and depth == 0:
            demangled = demangled[:i]
            break
    return demangled[5:] if demangled.startswith("void ") else demangled


def kernels(path):
    out = subprocess.run([CUOBJDUMP, "-sass", path], capture_output=True, text=True, check=True).stdout
    mangled, bodies, body = [], [], None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            mangled.append(m.group(1))
            body = []
            bodies.append(body)
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if body is not None and m:
            body.append(ANON.sub("ANON", re.sub(r"\s+", " ", m.group(1))))
    names = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.splitlines()
    ks = {}
    for n, b in zip(names, bodies):
        k = short_name(n.replace("(anonymous namespace)", "ANON"))
        if k in ks:
            raise SystemExit("two kernels named %s in %s" % (k, path))
        ks[k] = b
    return ks


def main(argv):
    if len(argv) != 3:
        raise SystemExit(__doc__)
    a, b = kernels(argv[1]), kernels(argv[2])
    same, diff, missing, merged = [], [], [], []
    for k in sorted(a):
        if k in b:
            (same if a[k] == b[k] else diff).append(k)
        elif k in RENAMES and RENAMES[k] in b:
            merged.append(k)
        else:
            missing.append(k)
    print("parent kernels: %d  branch kernels: %d" % (len(a), len(b)))
    print("identical under the same name: %d" % len(same))
    for k in same:
        print("  %s" % k)
    print("merged into another kernel: %d" % len(merged))
    for k in merged:
        n = RENAMES[k]
        verdict = "identical" if a[k] == b[n] else "different (%d -> %d instructions)" % (len(a[k]), len(b[n]))
        print("  %-26s -> %-34s %s" % (k, n, verdict))
    print("different under the same name: %d" % len(diff))
    for k in diff:
        print("  %s (%d -> %d instructions)" % (k, len(a[k]), len(b[k])))
    print("only in the parent: %d" % len(missing))
    for k in missing:
        print("  %s" % k)
    new = sorted(set(b) - set(a) - {RENAMES[k] for k in merged})
    print("only in the branch: %d" % len(new))
    for k in new:
        print("  %s" % k)
    return 0 if not diff and not missing else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv))
