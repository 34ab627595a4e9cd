"""Host-side pieces of bench.py that do not need a GPU: the read generators (SURVEY §8(d) config 2: 0.2 %
substitutions, 0.02 % indels), the stage -> kernel attribution of the roofline, the usable-CPU count, the output dump."""
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
import helpers as H
from vg_b200 import synth


def test_generators_produce_the_configured_error_model():
    g = synth.make_variant_graph(length=100000, n_snp=160, n_ins=20, n_del=20, n_haps=8, seed=5)
    index = g.build_index()
    n_pairs = 3000
    for reads, quals in (bench.simulate_pairs_numpy(g, n_pairs, 22), tuple(t.numpy() for t in bench.simulate_pairs_torch(g, n_pairs, 22, torch.device("cpu")))):
        assert reads.shape == (2 * n_pairs, bench.READ_LEN) and (quals == 30).all()
        res = H.oracle_map_paired(index, reads, quals, H.paired_params(bench.FRAG_MEAN, bench.FRAG_SD), threads=8)
        scores = res[0]["score"]
        assert (res[0]["flags"] & 1).mean() > 0.995
        clean = (scores == 160).mean()                    # no error at all: (1 - 0.002)^150 * (1 - 0.0296) = 0.72
        assert 0.66 < clean < 0.78
        gapped = np.isin(scores, (153, 154)).mean()       # exactly one 1-bp indel and nothing else: ~0.022
        assert 0.012 < gapped < 0.035
        assert res[4]["tail_dps"] > 0


def test_align_stage_split_names_the_seed_kernel_as_dominant(tmp_path):
    kernel_ms, split = bench.split_align_stage([13.57, 11.80, 13.97, 0.30])
    assert split is not None and abs(sum(split.values()) - 1.0) < 1e-9
    assert int(np.argmax(kernel_ms)) == 0 and kernel_ms[2] < 13.97
    # no profile: the stage times are used as they are
    kernel_ms, split = bench.split_align_stage([1.0, 2.0, 3.0, 0.1], summary_path=tmp_path / "missing.json")
    assert split is None and kernel_ms.tolist() == [1.0, 2.0, 3.0, 0.1]


def test_usable_cpus_is_positive():
    n, note = bench.usable_cpus()
    assert n >= 1 and isinstance(note, str)


def test_dump_outputs_writes_the_sampled_records_dereferenced(tmp_path):
    """--dump-outputs: float64 arrays whose mappings and edits, split by n_mappings / n_edits, are each sampled read's path."""
    g = synth.make_variant_graph(length=20000, n_snp=30, n_ins=4, n_del=4, n_haps=4, seed=9)
    index = g.build_index()
    rs = synth.simulate_pairs(g, 40, sub_rate=0.01, seed=5, indel_rate=0.002)
    aln, maps, edits, status, _ = H.oracle_map_paired(index, rs.reads, rs.quals, H.paired_params(), threads=2)
    idx = np.array([0, 3, 4, 17, 79])
    bench.dump_outputs(tmp_path, idx, aln[idx], status[idx], aln[idx]["mapping_off"], aln[idx]["edit_off"],
                       lambda i: maps[i], lambda i: edits[i])
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["read_index"].tolist() == idx.tolist() and got["aln_score"].tolist() == aln[idx]["score"].tolist()
    m = e = 0
    for r, i in enumerate(idx):
        _, _, path = H.decode_alignment(aln[i], maps, edits)
        nm, ne = int(got["aln_n_mappings"][r]), int(got["aln_n_edits"][r])
        assert got["mapping_node"][m: m + nm].tolist() == [n for n, _, _ in path]
        assert got["mapping_offset"][m: m + nm].tolist() == [o for _, o, _ in path]
        assert got["edits"][e: e + ne].tolist() == edits[int(aln[i]["edit_off"]): int(aln[i]["edit_off"]) + ne].tolist()
        m, e = m + nm, e + ne
    assert m == len(got["mapping_node"]) and e == len(got["edits"]) and m > 0 and e > 0
    # the sample is fixed: the same reads whatever the run
    s = bench.dump_sample(10_000_000)
    assert len(s) == bench.DUMP_READS and (np.diff(s) > 0).all() and (s == bench.dump_sample(10_000_000)).all()
    assert bench.dump_sample(100).tolist() == list(range(100))
