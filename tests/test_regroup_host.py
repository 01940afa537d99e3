"""CPU side of group births and deaths (dist_b200_regroup_batch): the numpy reference of the compaction, the Python
host mirrors following a remap, and the C++ mirror's regroup methods (compiled, linked and run without a device)."""
import os
import subprocess

import numpy as np

import regroup_ref as ref
from distributions_b200 import models

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_compaction_against_a_loop():
    rng = np.random.default_rng(0)
    for G in (1, 2, 5, 33, 1024, 2500):
        for n_empty in (1, 3):
            sizes = rng.integers(0, 4, G).astype(np.int32)
            rm, counts, G_new = ref.remap(sizes, n_empty)
            nxt, want_rm, want_counts = 0, [], []
            for g in range(G):
                if sizes[g] > 0:
                    want_rm.append(nxt)
                    want_counts.append(sizes[g])
                    nxt += 1
                else:
                    want_rm.append(-1)
            assert rm.tolist() == want_rm and counts.tolist() == want_counts + [0] * n_empty and G_new == nxt + n_empty
            assign = rng.integers(-2, G + 2, 1000).astype(np.int32)
            got = ref.relabel(assign, rm)
            for a, b in zip(assign, got):
                assert b == (a if a < 0 else (-1 if a >= G else want_rm[a]))
            stats = rng.integers(0, 9, (G, 3))
            out = ref.compact(stats, sizes, n_empty)
            assert out.shape == (G_new, 3)
            assert np.array_equal(out[:nxt], stats[sizes > 0]) and not out[nxt:].any()


def replay(counts, n_empty):
    """the per-value bookkeeping the batch replaces: remove_group (swap-with-last) of every empty group, then
    add_group until n_empty empty groups exist; each group is tracked by a label so that the result can be compared"""
    labels, c = list(range(len(counts))), list(counts)
    g = 0
    while g < len(c):
        if c[g] == 0:
            c[g], labels[g] = c[-1], labels[-1]
            c.pop()
            labels.pop()
        else:
            g += 1
    return dict(zip(labels, c)), len(c) + n_empty


def test_clustering_mirror_against_replay():
    rng = np.random.default_rng(1)
    for trial in range(50):
        G = int(rng.integers(1, 40))
        counts = rng.integers(0, 3, G).tolist()
        for Prior, model in ((models.PitmanYor, models.PitmanYor(1.0, 0.1)), (models.LowEntropy, models.LowEntropy(100))):
            mix = Prior.Mixture(None)
            mix.counts = [1] * G  # overwritten by counts=
            n_empty = int(rng.integers(1, 4))
            rm = mix.regroup(n_empty, counts=counts)
            survivors, G_replay = replay(counts, n_empty)
            assert len(mix) == G_replay
            assert {old: counts[old] for old in range(G) if rm[old] >= 0} == survivors
            assert [mix.counts[rm[old]] for old in sorted(survivors)] == [survivors[old] for old in sorted(survivors)]
            assert list(rm[rm >= 0]) == list(range(len(survivors)))  # survivors keep their order
            assert mix.empty_groupids == set(range(len(survivors), G_replay))
            assert mix.sample_size == sum(counts)


def test_id_tracker_against_replay():
    rng = np.random.default_rng(2)
    for trial in range(50):
        t = models.MixtureIdTracker(int(rng.integers(1, 30)))
        for _ in range(int(rng.integers(0, 10))):  # some churn first, so packed != global
            if rng.random() < 0.5 and t.packed_size() > 1:
                t.remove_group(int(rng.integers(t.packed_size())))
            else:
                t.add_group()
        sizes = rng.integers(0, 3, t.packed_size())
        before = [t.packed_to_global(p) for p in range(t.packed_size())]
        n_global = t.global_size()
        rm, _, G_new = ref.remap(sizes, 2)
        t.regroup(rm, 2)
        alive = [before[p] for p in range(len(before)) if sizes[p] > 0]
        assert t.packed_size() == G_new and t.global_size() == n_global + 2
        assert [t.packed_to_global(p) for p in range(G_new)] == alive + [n_global, n_global + 1]
        for p, glob in enumerate(alive):
            assert t.global_to_packed(glob) == p
        for p in range(len(before)):
            if sizes[p] == 0:
                assert before[p] not in t.global_to_packed_


def compile_regroup_api(out):
    """tests/cpp/test_regroup_api.cc against the library (and the CUDA runtime, for its device buffers in "gpu" mode)"""
    from distributions_b200 import build
    build.build()
    lib_dir = os.path.join(ROOT, "distributions_b200", "lib")
    cuda = os.path.dirname(os.path.dirname(build.NVCC))
    subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(cuda, "include"),
                    os.path.join(ROOT, "tests", "cpp", "test_regroup_api.cc"), "-o", out, "-L" + lib_dir, "-ldist_b200",
                    "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + lib_dir, "-Wl,-rpath," + os.path.join(cuda, "lib64")], check=True)
    return out


def test_cpp_mirror_regroup(tmp_path):
    exe = compile_regroup_api(str(tmp_path / "test_regroup_api"))
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr
