#!/usr/bin/env python
"""Kernel, memset and copy order per stream of the stacks' C calls, to compare two builds of libfegnn.so.

    FEGNN_LIB=<other build> python tools/forward_stack_launches.py record other.json
    python tools/forward_stack_launches.py record this.json
    python tools/forward_stack_launches.py compare other.json this.json > profiles/forward_stack_launches.txt

`record` runs each case below once to warm up, then once under torch.profiler with CUDA activities, and keeps per stream
the names of the kernels, memsets and copies in device order (streams numbered by first appearance).  It also keeps x and
Z of the deterministic forward-only stack on seeded inputs in fp32 and tf32 precision (in <json>.pt), which `compare`
checks bit for bit.  One build per process: the library is loaded at import."""
import json
import os
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.gpu_util import build_gpu_model, make_graph_case  # noqa: E402
from fastegnn_b200 import CsrGraph, FastEGNN, FastRF, _lib  # noqa: E402

DEV = "cuda:0"
WATER3D = dict(seed=3, sizes=[8000], deg=22, C=3, gravity=[0, -1, 0])       # Water-3D size: the forward-only ring of 4
LARGE = dict(seed=12, sizes=[100_000], deg=8, C=8)                          # > 65 536 nodes: the forward-only single block
# name -> (graph, layers, FastRF, what runs); train: forward + backward, rc: with recompute, backward twice over one
# forward (the second with FEGNN_F_REBUILD_ALL); infer: the forward-only stack (eval, no_grad); prebuilt: a CsrGraph
# built ahead (no pending sort); det: under torch.use_deterministic_algorithms(True)
CASES = {
    "train water3d L4": (WATER3D, 4, False, "train"),
    "train recompute water3d L4, two backwards": (WATER3D, 4, False, "rc"),
    "forward-only water3d L4 (ring)": (WATER3D, 4, False, "infer"),
    "forward-only water3d L6 (ring refills)": (WATER3D, 6, False, "infer"),
    "forward-only 100k L4 (one block), prebuilt graph": (LARGE, 4, False, "prebuilt"),
    "FastRF train water3d L4": (WATER3D, 4, True, "train"),
    "FastRF forward-only water3d L4": (WATER3D, 4, True, "infer"),
    "deterministic forward-only water3d L4 (ring)": (WATER3D, 4, False, "det"),
    "deterministic forward-only 100k L4 (one block)": (LARGE, 4, False, "det"),
    "deterministic FastRF forward-only water3d L4": (WATER3D, 4, True, "det"),
}


def setup(graph, L, rf):
    kw = dict(graph)
    cfg, params, inp = make_graph_case(kw.pop("seed"), kw.pop("sizes"), kw.pop("deg"), kw.pop("C"), L=L, **kw)
    if rf:
        torch.manual_seed(graph["seed"])
        m = FastRF(node_feat_nf=cfg.node_feat_nf, node_attr_nf=0, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
                   virtual_channels=cfg.virtual_channels, device=DEV, n_layers=L, gravity=cfg.gravity)
    else:
        m = build_gpu_model(cfg, params, DEV)
    return m, {k: v.to(DEV) for k, v in inp.items()}


def runner(m, t, how):
    def args(edge_index):
        return dict(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=t["node_vel"], edge_index=edge_index,
                    data_batch=t["data_batch"], loc_mean=t["loc_mean"])
    if how in ("train", "rc"):
        m.train()
        m.recompute = how == "rc"

        def run():
            x, Z = m(**args(t["edge_index"]), edge_attr=t["edge_attr"])
            loss = (x * t["wx"]).sum() + (Z * t["wz"]).sum()
            n = 2 if how == "rc" else 1
            for i in range(n):
                loss.backward(retain_graph=i + 1 < n)
        return run
    m.eval()
    if how == "prebuilt":
        g = CsrGraph(t["edge_index"], t["data_batch"], t["edge_attr"], int(t["loc_mean"].size(0)))
        return lambda: m(**args(g))
    return lambda: m(**args(t["edge_index"]), edge_attr=t["edge_attr"])


def trace(fn):
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path))["traceEvents"]
    rows = sorted((e["ts"], e["args"]["stream"], e["name"]) for e in events
                  if e.get("cat") in ("kernel", "gpu_memset", "gpu_memcpy"))
    label, out = {}, {}
    for _, s, name in rows:
        label.setdefault(s, f"stream {len(label)}")
        out.setdefault(label[s], []).append(name)
    return out


def record(path):
    det_on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    launches, outputs = {}, {}
    for name, (graph, L, rf, how) in CASES.items():
        m, t = setup(graph, L, rf)
        torch.use_deterministic_algorithms(how == "det")
        try:
            fn = runner(m, t, how)
            if how in ("train", "rc"):
                launches[name] = trace(fn)
                continue
            with torch.no_grad():
                launches[name] = trace(fn)
                if how == "det":
                    for prec in ("fp32", "tf32"):
                        _lib.set_precision(prec)
                        x, Z = fn()
                        outputs[f"{name} [{prec}]"] = (x.cpu(), Z.cpu())
        finally:
            _lib.set_precision("tf32")
            torch.use_deterministic_algorithms(det_on, warn_only=warn_only)
            _lib.set_mode("deterministic", 0)
        print(f"{name}: " + ", ".join(f"{s} {len(v)}" for s, v in launches[name].items()), flush=True)
    json.dump(dict(lib=_lib.LIB_PATH, launches=launches), open(path, "w"), indent=1)
    torch.save(outputs, path + ".pt")


def compare(path_a, path_b):
    a, b = json.load(open(path_a)), json.load(open(path_b))
    oa, ob = torch.load(path_a + ".pt"), torch.load(path_b + ".pt")
    same = True
    print(f"# A: {os.path.basename(path_a)}  B: {os.path.basename(path_b)}")
    print("# per case and stream: kernels, memsets and copies of one call in device order (streams numbered by first use)")
    for name in CASES:
        la, lb = a["launches"][name], b["launches"][name]
        ok = la == lb
        same &= ok
        print(f"{'identical' if ok else 'DIFFERENT'}  {name}: " + ", ".join(f"{s} {len(v)}" for s, v in lb.items()))
        if not ok:
            for s in sorted(set(la) | set(lb)):
                if la.get(s) != lb.get(s):
                    print(f"  {s}\n    A: {la.get(s)}\n    B: {lb.get(s)}")
    for name in sorted(oa):
        ok = all(torch.equal(p, q) for p, q in zip(oa[name], ob[name]))
        same &= ok
        print(f"{'bitwise  ' if ok else 'DIFFERENT'}  x, Z of {name}")
    print("\n# the listing of B, case by case")
    for name in CASES:
        print(f"\n## {name}")
        for s, names in b["launches"][name].items():
            print(f"{s}:")
            print("\n".join(f"  {n}" for n in names))
    return 0 if same else 1


if __name__ == "__main__":
    if sys.argv[1:2] == ["record"] and len(sys.argv) == 3:
        record(sys.argv[2])
    elif sys.argv[1:2] == ["compare"] and len(sys.argv) == 4:
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
