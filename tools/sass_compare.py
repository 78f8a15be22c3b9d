#!/usr/bin/env python
"""Compare the SASS of two builds of spsg_raycast.cu function by function, instruction offsets and encodings stripped
(no GPU needed).  The backward gather's template gained parameters (kUpstream, then kViewNormals, then kSegments); its old
instantiations <kFused, kViews> and <kFused, kUpstream, kViews> are matched with kUpstream / kViewNormals / kSegments /
kGenericSem false.  The forward kernel's <kLoss, kSmemMaps, kWarps> likewise with <kLoss, kSmemMaps, kWarps, kViewNormals =
false, kGenericSem = false, kLabels = false, kEval = false>, and the stand-alone loss kernels (losses2d_forward/backward/det_kernel) with their
<kGenericSem = false> instantiations.  The compaction kernels of spsg_sparsify.cu gained the SDF
element type: the plain sparsify_count_kernel and sparsify_write_kernel<kIndexed> are matched with their <float>
instantiations.

    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -I include -Xptxas -v -cubin \\
         <package>/csrc/spsg_raycast.cu -o after.cubin          # and the same on the older tree -> before.cubin
                                                                # (likewise spsg_sparsify.cu)
    python tools/sass_compare.py before.cubin after.cubin
"""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def functions(cubin):
    out = subprocess.check_output([CUOBJDUMP, "-sass", cubin], text=True)
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
            continue
        if cur is None:
            continue
        line = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)     # instruction offsets
        line = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", line)    # encodings
        line = re.sub(r"_ZN\w+", "SYM", line).strip()      # branch targets / callees named by their mangled symbol
        if line:
            res[cur].append(line)
    return res


def key(name):
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]{8}", "", name)  # the anonymous namespace's per-build tag
    m = re.search(r"backward_gather_kernelI(Lb[01]E)(Lb[01]E)?(Li\dE)(Lb[01]E)?(Lb[01]E)?(Lb[01]E)?E", name)
    if m:
        return "backward_gather_kernel" + m.group(1) + (m.group(2) or "Lb0E") + m.group(3) + (m.group(4) or "Lb0E") + \
            (m.group(5) or "Lb0E") + (m.group(6) or "Lb0E")
    m = re.search(r"raycast_forward_kernelI(Lb[01]ELb[01]ELi\d+E)(Lb[01]E)?(Lb[01]E)?(Lb[01]E)?(Lb[01]E)?E", name)
    if m:
        return "raycast_forward_kernel" + m.group(1) + (m.group(2) or "Lb0E") + (m.group(3) or "Lb0E") + \
            (m.group(4) or "Lb0E") + (m.group(5) or "Lb0E")
    m = re.search(r"(losses2d_(?:forward|backward|det)_kernel)(?:ILb([01])EE)?", name)
    if m:
        return "%s<%s>" % (m.group(1), m.group(2) or "0")
    m = re.search(r"sparsify_count_kernel(?:I([a-z])EEv)?", name)
    if m:
        return "sparsify_count_kernel<%s>" % (m.group(1) or "f")
    m = re.search(r"sparsify_write_kernelI([a-z])?(Lb[01]E)E", name)
    if m:
        return "sparsify_write_kernel<%s,%s>" % (m.group(1) or "f", m.group(2))
    return name


def main(before, after):
    a = {key(n): v for n, v in functions(before).items()}
    b = {key(n): v for n, v in functions(after).items()}
    differing = 0
    for k in sorted(a):
        if k not in b:
            print("only in %s: %s" % (before, k))
            differing += 1
        elif a[k] != b[k]:
            diff = sum(x != y for x, y in zip(a[k], b[k])) + abs(len(a[k]) - len(b[k]))
            print("differs: %s (%d of %d lines)" % (k, diff, len(a[k])))
            differing += 1
    print("%d functions compared, %d identical, %d differing; new: %s" % (
        len(a), len(a) - differing, differing, ", ".join(sorted(k for k in b if k not in a)) or "none"))
    return 1 if differing else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
