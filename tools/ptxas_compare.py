"""Kernel-by-kernel comparison of two `-Xptxas -v` logs of libfegnn.so (a parent build and this one).

Make each log from a checkout of the build it describes (nvcc prints the listing on stderr):

    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -shared -Xptxas -v \\
        fastegnn_b200/csrc/api.cu -o /tmp/libfegnn.so 2> ptxas.log

    python tools/ptxas_compare.py parent.log this.log > profiles/input_grads_ptxas.txt

Kernels are matched by mangled name, a name the parent lacks after renamings that do not change the code: the anonymous
namespace of api.cu (its hash depends on the source path), the `kEa = false` instantiations of edge_bwd_kernel /
edge_bwd_tc4_kernel and the `kDet = false` instantiations of the forward kernels (edge_fwd_kernel, edge_fwd_tc_kernel,
virtual_fwd_kernel, virtual_fwd_tc_kernel, node_h_z_kernel), the `kSaved = false` instantiations of virtual_fwd_kernel,
virtual_fwd_tc_kernel and node_h_fwd_tc_kernel, and the `kLive = false` instantiations of the kernels that walk edges
(LIVE_ADDED), which are a parent's untemplated (resp. one-parameter fewer) kernels.  Every kernel of both builds is listed with its resource
lines (stack frame, spills, registers, barriers, shared memory; constant-bank sizes are left out)."""
import re
import sys

ANON = re.compile(r"_GLOBAL__N__[0-9a-f]{8}_6_api_cu_[0-9a-f]{8}")


def parse(path):
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            cur = ANON.sub("_GLOBAL__N_api_cu", m.group(1))
            out[cur] = []
            continue
        if cur and ("stack frame" in line or "Used " in line):
            out[cur].append(line.split("ptxas info    :")[-1].strip())
    return out


# a trailing bool template parameter (false) that a parent does not have: "kernelI<args>Lb0EEEv" -> "kernelI<args>EEv",
# and a kernel whose only template parameter it is: "kernelILb0EEEvNS_" -> "kernelENS_"
BOOL_ADDED = ("edge_bwd_kernel", "edge_bwd_tc4_kernel", "edge_fwd_kernel", "edge_fwd_tc_kernel", "virtual_fwd_kernel",
              "virtual_fwd_tc_kernel", "node_h_z_kernel", "node_h_fwd_tc_kernel")
# a second trailing bool (the kSaved = false forms of the recompute, FEGNN_F_RECOMPUTE) after the kDet one
BOOL2_ADDED = ("virtual_fwd_kernel", "virtual_fwd_tc_kernel")
# the kLive = false forms of the kernels that walk edges (FEGNN_F_LIVE_EDGES): a trailing bool after the parent's parameters
LIVE_ADDED = ("edge_fwd_kernel", "edge_fwd_tc_kernel", "edge_bwd_kernel", "edge_bwd_tc4_kernel", "edge_det_fixup_kernel")


def to_parent(name, parent):
    if name in parent:
        return name
    for k in LIVE_ADDED:
        if f"{len(k)}{k}I" in name:
            trimmed = name.replace(f"{k}ILb0EEEvNS_", f"{k}ENS_")
            trimmed = re.sub(rf"({k}I(?:L[ib]\d+E)+)Lb0EEEv", r"\1EEv", trimmed)
            if trimmed != name:
                return to_parent(trimmed, parent)
    for k in BOOL2_ADDED:
        if f"{len(k)}{k}I" in name:
            trimmed = re.sub(rf"({k}I(?:L[ib]\d+E)+)Lb0EEEv", r"\1EEv", name)
            if trimmed in parent:
                return trimmed
    for k in BOOL_ADDED:
        if f"{len(k)}{k}I" in name:
            name = name.replace(f"{k}ILb0EEEvNS_", f"{k}ENS_")
            return re.sub(rf"({k}I(?:Li\d+E)+)Lb0EEEv", r"\1EEv", name)
    return name


def main(parent_log, this_log):
    a, b = parse(parent_log), parse(this_log)
    matched = {k: to_parent(k, a) for k in b if to_parent(k, a) in a}
    same = sum(a[p] == b[k] for k, p in matched.items())
    new = [k for k in b if k not in matched]
    gone = [p for p in a if p not in set(matched.values())]
    print(f"{same} kernels with identical -Xptxas -v lines, {len(matched) - same} changed, {len(new)} new, {len(gone)} gone")
    for k in sorted(new):
        print(f"NEW      {k} {b[k]}")
    for p in sorted(gone):
        print(f"GONE     {p} {a[p]}")
    for k in sorted(matched):
        p = matched[k]
        tag = "same" if a[p] == b[k] else "CHANGED"
        print(f"{tag:8} parent {p} {a[p]}")
        print(f"{'':8} this   {k} {b[k]}")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
