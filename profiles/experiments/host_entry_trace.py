"""Copy and launch sequence of the host-buffer scoring entries, for every configuration of tests/test_gpu_host_entries.py.

Each configuration (feature list, output, chunking, buffers, zero-copy option) makes one host-entry call under
torch.profiler with CUDA activities.  The call's GPU activities are listed per stream, streams numbered by first
appearance within the call, each in start order: kernels by name, memcpys by kind and bytes, memsets by bytes.  The
sequence on one stream does not depend on timing, so two builds run with the same arguments can be compared line for
line (the interleaving across streams can, and is not listed).  Run on a B200:

    python profiles/experiments/host_entry_trace.py [--root TREE] --out trace.txt   # TREE: the tree whose library runs
    python profiles/experiments/host_entry_trace.py --diff parent.txt branch.txt     # summary of the differences

host_entry_trace.txt is that summary for the commit that gave the host entries one staging helper (branch) against its
parent: every difference is the per-row output of the one-compute-stream schedule (any niw feature, or dpd in a list or
under logp) coming back as one D2H copy per row chunk instead of one copy at the end.
"""
import argparse
import collections
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GPU_CATS = ("kernel", "gpu_memcpy", "gpu_memset")


def activity(e):
    a = e.get("args", {})
    if e["cat"] == "kernel":
        return "kernel %s" % e["name"]
    return "%s %d" % (e["name"], a.get("bytes", -1))


def calls(trace_events):
    """the GPU activities between consecutive marker kernels (torch fills on the caller's side), per call"""
    evs = sorted((e for e in trace_events if e.get("cat") in GPU_CATS), key=lambda e: e["ts"])
    out, cur = [], None
    for e in evs:
        if e["cat"] == "kernel" and "FillFunctor" in e["name"]:
            if cur is not None:
                out.append(cur)
            cur = [] if cur is None else None
            continue
        if cur is not None:
            cur.append(e)
    return out


def per_stream(evs):
    streams = collections.OrderedDict()
    for e in evs:
        streams.setdefault(e["args"].get("stream"), []).append(activity(e))
    return ["s%d %s" % (i, a) for i, acts in enumerate(streams.values()) for a in acts]


def trace(root, out_path):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, root)
    import torch
    from torch.profiler import ProfilerActivity, profile

    import test_gpu_host_entries as t
    from distributions_b200 import capi

    assert os.path.dirname(capi.__file__).startswith(os.path.abspath(root)), capi.__file__
    ctx = capi.Context(0)
    marker = torch.zeros(1, device="cuda", dtype=torch.int32)
    lines = ["device: %s" % torch.cuda.get_device_name(0)]
    for lst in t.LISTS:
        configs = [(out, ch, kind, zc) for (l, out) in t.CASES if l == lst for ch in t.CHUNKINGS for kind, zc in t.BUFFER_RUNS]
        # inputs, features, GP tables and scratch ready before the profiled calls
        for out, n in sorted({(out, t.CHUNKINGS[ch][0]) for out, ch, _, _ in configs}):
            t.run_host(ctx, t.setup(ctx, lst, n), out, "pageable", 0, 0)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for out, ch, kind, zc in configs:
                n, chunks = t.CHUNKINGS[ch]
                s = t.setup(ctx, lst, n)
                with t.buffers(ctx, s, out, kind) as (cols, u, dst):
                    ctx.set_option(capi.OPT_HOST_CHUNKS, chunks)
                    ctx.set_option(capi.OPT_HOST_ZEROCOPY, zc)
                    try:
                        torch.cuda.synchronize()
                        marker.fill_(1)
                        torch.cuda.synchronize()
                        t.call_host(ctx, s, out, cols, u, dst)
                        marker.fill_(2)
                        torch.cuda.synchronize()
                    finally:
                        ctx.set_option(capi.OPT_HOST_CHUNKS, 0)
                        ctx.set_option(capi.OPT_HOST_ZEROCOPY, 0)
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as fh:
                got = calls(json.load(fh)["traceEvents"])
        assert len(got) == len(configs), "%s: %d calls traced for %d configurations" % (lst, len(got), len(configs))
        for (out, ch, kind, zc), evs in zip(configs, got):
            lines.append("== %s %s %s %s zerocopy=%d" % (lst, out, ch, kind, zc))
            lines += ["  " + a for a in per_stream(evs)]
    ctx.close()
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


def parse(path):
    cfgs, cur = collections.OrderedDict(), None
    with open(path) as fh:
        for line in fh:
            if line.startswith("device: "):
                print("%s: %s" % (os.path.basename(path), line.strip()))
            elif line.startswith("== "):
                cur = cfgs.setdefault(line[3:].strip(), [])
            elif cur is not None:
                cur.append(line.strip())
    return cfgs


def diff(a_path, b_path):
    """configurations whose sequences are identical; the others, with what differs apart from the D2H copies and whether
    the D2H copies move the same bytes per stream"""
    a, b = parse(a_path), parse(b_path)
    assert list(a) == list(b), "the two traces list different configurations"
    same, other = 0, []
    for cfg in a:
        if a[cfg] == b[cfg]:
            same += 1
            continue
        d2h = lambda seq: [x for x in seq if " DtoH " in x]  # noqa: E731
        rest = lambda seq: [x for x in seq if " DtoH " not in x]  # noqa: E731
        def d2h_bytes(seq):
            tot = collections.Counter()
            for x in d2h(seq):
                tot[x.split()[0] + " " + x[x.index("("):x.index(")") + 1]] += int(x.split()[-1])
            return dict(tot)
        other.append((cfg, rest(a[cfg]) == rest(b[cfg]), d2h_bytes(a[cfg]) == d2h_bytes(b[cfg]), len(d2h(a[cfg])), len(d2h(b[cfg]))))
    print("configurations: %d, identical sequences: %d, different: %d" % (len(a), same, len(other)))
    ok = all(r and y for _, r, y, _, _ in other)
    print("every difference is in the D2H copies alone, with the same bytes per stream and kind: %s" % ("yes" if ok else "NO"))
    for cfg, r, y, na, nb in other:
        print("  %-60s D2H copies %d -> %d%s%s" % (cfg, na, nb, "" if r else ", OTHER ACTIVITIES DIFFER", "" if y else ", D2H BYTES DIFFER"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=ROOT, help="tree whose distributions_b200 (and built library) is traced")
    ap.add_argument("--out", help="trace file to write")
    ap.add_argument("--diff", nargs=2, metavar=("A", "B"), help="summarise the differences of two trace files")
    args = ap.parse_args()
    if args.diff:
        diff(*args.diff)
    else:
        trace(os.path.abspath(args.root), args.out)
