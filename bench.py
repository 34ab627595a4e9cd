#!/usr/bin/env python
"""bench.py — giraffe reads/sec on BASELINE.json configs[1] (1 Mbp / 1k-variant graph,
150 bp paired-end reads), one process per GPU.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the CPU restatement of vg giraffe
                                                           # (oracle/) on the box's host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's records as DIR/*.npy

A "step" is one pass of the mapping hot path over one batch of synthetic read pairs.
value  = whole-job reads/s with the reads already resident in HBM (device-pointer C-ABI entry,
         CUDA events on the launching stream);
e2e    = the same batch through the host-buffer C-ABI entry gb_map_paired_batch (pinned host
         memory, H2D of reads+qualities and D2H of the alignment records inside the timed region).
Rank 0 prints one JSON line.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

READ_LEN = 150
WORKLOAD = ("configs[1]: 1 Mbp random graph, 1k SNP+indel variants, 8 haplotypes, nodes <= 32 bp, k=29 w=11; "
            "150 bp paired-end reads, fragment N(400,50) forced, 0.2 % substitutions, 0.02 % indels (SURVEY §8(d) config 2)")
FRAG_MEAN, FRAG_SD = 400.0, 50.0
SUB_RATE = 0.002
INDEL_RATE = 0.0002        # per base, SURVEY.md §8(d) config 2; at most one 1-bp insertion or deletion per read, half each
GRAPH_SEED = 2


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------
# synthetic workload
# ---------------------------------------------------------------------------------------
def make_graph_and_index():
    from vg_b200 import synth
    t = time.time()
    g = synth.make_variant_graph(length=1_000_000, n_snp=800, n_ins=100, n_del=100, n_haps=8, seed=GRAPH_SEED)
    index = g.build_index(k=29, w=11)
    log(f"[bench] graph+index: {len(g.node_seqs)} nodes, {index.view.n_hits} minimizer hits, {time.time() - t:.1f}s")
    return g, index


def simulate_pairs_torch(g, n_pairs, seed, device):
    """GPU version of synth.simulate_pairs (inward 150 bp pairs, fragment N(400, 50), 0.2 % substitutions,
    0.02 % indels)."""
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    haps = [torch.from_numpy(h.copy()).to(device) for h in g.hap_seq]
    min_len = min(len(h) for h in haps)
    comp = torch.full((256,), ord("N"), dtype=torch.uint8, device=device)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    bases = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=device)
    reads = torch.empty((2 * n_pairs, READ_LEN), dtype=torch.uint8, device=device)
    ar = torch.arange(READ_LEN, device=device)
    CH = 250_000
    for c0 in range(0, n_pairs, CH):
        cn = min(CH, n_pairs - c0)
        hap = torch.randint(0, len(haps), (cn,), generator=gen, device=device)
        frag = torch.clamp(torch.round(torch.randn(cn, generator=gen, device=device) * FRAG_SD + FRAG_MEAN), min=READ_LEN).long()
        start = (torch.rand(cn, generator=gen, device=device) * (min_len - 1000)).long()
        flip = torch.rand(cn, generator=gen, device=device) < 0.5
        # one 1-bp indel per read with probability 1 - (1 - INDEL_RATE)^L: a deletion skips haplotype base p,
        # an insertion puts a random base at p and shifts the rest (both in haplotype coordinates of the window)
        def indel_events():
            hit = torch.rand(cn, generator=gen, device=device) < 1.0 - (1.0 - INDEL_RATE) ** READ_LEN
            kind = torch.where(hit, torch.randint(1, 3, (cn,), generator=gen, device=device), torch.zeros(cn, dtype=torch.long, device=device))
            pos = torch.randint(1, READ_LEN - 1, (cn,), generator=gen, device=device)
            ins = bases[torch.randint(0, 4, (cn,), generator=gen, device=device)]
            off = (kind[:, None] == 1).long() * (ar[None, :] >= pos[:, None]).long() - (kind[:, None] == 2).long() * (ar[None, :] > pos[:, None]).long()
            return kind, pos, ins, off
        kind_l, pos_l, ins_l, off_l = indel_events()
        kind_r, pos_r, ins_r, off_r = indel_events()
        left = torch.empty((cn, READ_LEN), dtype=torch.uint8, device=device)
        right = torch.empty((cn, READ_LEN), dtype=torch.uint8, device=device)
        for h in range(len(haps)):
            sel = (hap == h).nonzero(as_tuple=True)[0]
            if sel.numel() == 0:
                continue
            rs = start[sel] + frag[sel] - READ_LEN
            lwin = haps[h][start[sel, None] + ar[None, :] + off_l[sel]]
            rwin = haps[h][rs[:, None] + ar[None, :] + off_r[sel]]
            lwin = torch.where((kind_l[sel, None] == 2) & (ar[None, :] == pos_l[sel, None]), ins_l[sel, None], lwin)
            rwin = torch.where((kind_r[sel, None] == 2) & (ar[None, :] == pos_r[sel, None]), ins_r[sel, None], rwin)
            left[sel] = lwin
            right[sel] = comp[rwin.long()].flip(1)
        m1 = torch.where(flip[:, None], right, left)
        m2 = torch.where(flip[:, None], left, right)
        reads[2 * c0: 2 * (c0 + cn): 2] = m1
        reads[2 * c0 + 1: 2 * (c0 + cn): 2] = m2
    # substitutions
    for c0 in range(0, 2 * n_pairs, 1_000_000):
        blk = reads[c0: c0 + 1_000_000]
        mask = torch.rand(blk.shape, generator=gen, device=device) < SUB_RATE
        idx = mask.nonzero(as_tuple=True)
        if idx[0].numel():
            old = blk[idx]
            code = (old == ord("C")).long() + 2 * (old == ord("G")).long() + 3 * (old == ord("T")).long()
            new = bases[(code + torch.randint(1, 4, code.shape, generator=gen, device=device)) % 4]
            blk[idx] = new
    quals = torch.full_like(reads, 30)
    return reads, quals


def simulate_pairs_numpy(g, n_pairs, seed):
    from vg_b200 import synth
    rs = synth.simulate_pairs(g, n_pairs, length=READ_LEN, frag_mean=FRAG_MEAN, frag_sd=FRAG_SD, sub_rate=SUB_RATE, indel_rate=INDEL_RATE, seed=seed)
    return rs.reads, rs.quals


# ---------------------------------------------------------------------------------------
# helpers

def split_align_stage(last_stage, summary_path=None):
    """Per-kernel times from the four stage timers: the align stage (index 2) is three launches, so its dominant
    kernel (the warp-per-pair align_kernel_pe) gets the stage time times its share in the committed ncu launch list.
    Returns (kernel_ms[4], split or None)."""
    kernel_ms = np.array(last_stage, dtype=np.float64)
    align_split = None
    try:
        kern = json.loads(Path(summary_path or (ROOT / "profiles" / "ncu_summary_r01.json")).read_text())["kernels"]
        parts = {k: float(kern[k]["total_ms"]) for k in ("align_fast_kernel_pe", "align_kernel_pe", "align_kernel_pe<rescue>") if k in kern and "total_ms" in kern[k]}
        if "align_kernel_pe" in parts and sum(parts.values()) > 0:
            align_split = {k: v / sum(parts.values()) for k, v in parts.items()}
            kernel_ms[2] = float(last_stage[2]) * align_split["align_kernel_pe"]
    except Exception:
        pass
    return kernel_ms, align_split

# ---------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cpus():
    """Host CPUs this process may actually use: min(affinity, cgroup cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    note = f"{n} logical CPUs"
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            q = max(1, int(int(quota) / int(period)))
            if q < n:
                note = f"cgroup cpu.max quota {q} of {n} logical CPUs"
                n = q
    except Exception:
        pass
    return n, note


def oracle_library(native=True):
    """liboracle.so, rebuilt with -march=native for the host that runs the benchmark when gcc is available (test
    infrastructure; only the cpu_baseline leg and --impl reference use it).  The native build goes to a temporary
    directory: the benchmark writes nothing into the source tree."""
    import helpers as H
    if native:
        try:
            with tempfile.TemporaryDirectory(prefix="bench_oracle_") as tmp:
                so = Path(tmp) / "liboracle.so"
                srcs = sorted(str(p) for p in (ROOT / "oracle").glob("*.cpp"))
                cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
                subprocess.run([cxx, "-O3", "-march=native", "-std=c++17", "-fPIC", "-fopenmp", "-shared", "-o", str(so)] + srcs,
                               check=True, capture_output=True, cwd=str(ROOT / "oracle"))
                H._oracle = None
                lib = C.CDLL(str(so))          # stays mapped after the directory is removed
            H._oracle = lib
            H.oracle_lib_configure(lib)
            return lib, "-O3 -march=native"
        except Exception as e:  # fall back to the prebuilt generic build
            log(f"[bench] native oracle build failed ({e}); using the prebuilt library")
            H._oracle = None
    return H.oracle_lib(), "-O3 (generic)"


def cpu_map_rate(index, reads_np, quals_np, params, threads, target_seconds=15.0):
    """reads/s of the CPU restatement over a bounded sample; output buffers are allocated and touched
    once, and the thread count is the best of {all logical CPUs, physical cores, 32, 16}."""
    import helpers as H
    n_total = reads_np.shape[0]
    probe = min(n_total, 400_000)
    probe -= probe % 2
    out = H.oracle_out_buffers(n_total, params)
    H.oracle_map_paired(index, reads_np[:probe], quals_np[:probe], params, threads=threads, out=out)      # warm
    best = (0.0, threads)
    for th in sorted({threads, max(1, threads // 2), 2 * threads}, reverse=True):
        t = time.time()
        H.oracle_map_paired(index, reads_np[:probe], quals_np[:probe], params, threads=th, out=out)
        r = probe / max(time.time() - t, 1e-6)
        if r > best[0]:
            best = (r, th)
    rate, th = best
    sample = int(min(n_total, max(probe, rate * target_seconds)))
    sample -= sample % 2
    t = time.time()
    res = H.oracle_map_paired(index, reads_np[:sample], quals_np[:sample], params, threads=th, out=out)
    dt = time.time() - t
    return sample / dt, sample, dt, res, th


DUMP_READS = 65536          # --dump-outputs: records of this many reads of the last step (a fixed, seeded sample of a larger step)
DUMP_MAX_BYTES = 64 << 20


def dump_sample(n_reads):
    """Indices of the reads whose records --dump-outputs writes: every read of a small step, else a fixed seeded sample."""
    if n_reads <= DUMP_READS:
        return np.arange(n_reads, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n_reads, DUMP_READS, replace=False)).astype(np.int64)


def pool_ranges(starts, counts):
    """The concatenation of arange(s, s + c) over the pairs of starts and counts."""
    starts, counts = starts.astype(np.int64), counts.astype(np.int64)
    return np.repeat(starts - np.cumsum(counts) + counts, counts) + np.arange(int(counts.sum()), dtype=np.int64)


def dump_outputs(out_dir, reads, aln, status, map_start, edit_start, take_maps, take_edits):
    """Write the records of the reads `reads` as out_dir/<name>.npy, float64 (exact for every field).
    aln and status are those reads' headers (read_id as an index into the step's reads) and item status; map_start and
    edit_start are where each read's mappings and edits begin in the step's pools, and take_maps / take_edits fetch pool
    entries by index.  Mappings and edits are written dereferenced and concatenated in read order (n_mappings and n_edits
    split them), so the files do not depend on how a build lays out its pools."""
    maps = take_maps(pool_ranges(map_start, aln["n_mappings"]))
    edits = take_edits(pool_ranges(edit_start, aln["n_edits"]))
    arrays = {"read_index": reads, "status": status, "edits": edits}
    for f in ("read_id", "score", "mapq", "flags", "n_mappings", "n_edits", "mapq_uncapped", "mapq_explored_cap"):
        arrays[f"aln_{f}"] = aln[f]
    for f in ("node", "offset", "n_edits"):
        arrays[f"mapping_{f}"] = maps[f]
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, v in arrays.items():
        np.save(out / f"{k}.npy", v)
    log(f"[bench] --dump-outputs: {len(reads)} reads, {len(maps)} mappings, {len(edits)} edits, {total} bytes in {out}")


def algorithmic_bytes_per_read(L, counters, n_reads_sample, mappings_per_read, edits_per_read):
    """SURVEY.md §8(d): B(read) = 2L + 16M + 24H + X(L + 16 ceil(L/32) + 16) + T(S_t + 16 N_t) + 32 + 8P + 4E."""
    M = counters["minimizers"] / n_reads_sample
    Hh = counters["seeds"] / n_reads_sample
    X = counters["extend_calls"] / n_reads_sample
    T = counters["tail_dps"] / n_reads_sample
    St = counters["tail_bases"] / max(counters["tail_dps"], 1)
    Nt = counters["tail_nodes"] / max(counters["tail_dps"], 1)
    per_kernel = {
        # the seeding kernel reads the bases, one 16-B table cell per minimizer and one 24-B hit per seed
        "seed_kernel_pe": L + 16 * M + 24 * Hh,
        # per gapless extension: L graph bases and 16 B per node record (+1 node)
        "extend_kernel": X * (L + 16 * -(-L // 32) + 16),
        # align stage: qualities (MAPQ cap), tail subgraphs, the output record
        "align_kernel_pe": L + T * (St + 16 * Nt) + 32 + 8 * mappings_per_read + 4 * edits_per_read,
        "compact": 0.0,
    }
    B = 2 * L + 16 * M + 24 * Hh + X * (L + 16 * -(-L // 32) + 16) + T * (St + 16 * Nt) + 32 + 8 * mappings_per_read + 4 * edits_per_read
    return B, {"M": round(M, 2), "H": round(Hh, 2), "X": round(X, 3), "T": round(T, 4), "S_t": round(St, 1), "N_t": round(Nt, 1),
               "P": round(mappings_per_read, 2), "E": round(edits_per_read, 2)}, per_kernel


def secondary_workloads(ordinal, n=200_000, check=10_000):
    """BASELINE.json configs[3], configs[4] and the single-end path on the configs[1] graph, as secondary fields of the bench
    line (not the metric): kernel-time reads/s of one gb_map_batch call (best of 2), per-kernel times, and a parity count of the
    first `check` reads against the CPU restatement."""
    import helpers as H
    from vg_b200 import capi, synth
    out = {}
    threads, _ = usable_cpus()
    for name, make_graph, kw in [
        ("configs[3] branchy graph (8 bp nodes, 4-way bubbles), 150 bp SE", lambda: synth.make_branchy_graph(), dict(length=150, sub_rate=0.005, seed=44)),
        ("configs[4] 250 bp SE, 5 % errors (tail DP)", lambda: synth.make_variant_graph(), dict(length=250, sub_rate=0.03, ins_rate=0.01, del_rate=0.01, seed=55)),
        ("configs[1] graph, 150 bp SE", lambda: synth.make_variant_graph(), dict(length=150, sub_rate=0.002, seed=23)),
    ]:
        g = make_graph(); index = g.build_index()
        rs = synth.simulate_reads(g, n, **kw)
        dev = capi.Device(index, ordinal)
        rbuf, qbuf, read_off = H.pack_reads(rs.reads, rs.quals)
        best = None
        for _ in range(2):
            got = dev.map_arrays(rbuf, qbuf, read_off)
            best = dev.kernel_ms() if best is None else min(best, dev.kernel_ms())
        kern = {}
        for k, v in dev.kernel_times():
            kern[k] = round(kern.get(k, 0.0) + v, 3)
        plan = dev.plan_stats()
        want = H.oracle_map(index, rs.reads[:check], rs.quals[:check], threads=threads)
        bad = H.compare_alignments(got, want, check)
        cells = int(want[4]["tail_cells"]) * n // check
        out[name] = {"reads": n, "reads_per_s": n / (best / 1e3), "kernel_ms": best, "kernel_ms_by_kernel": kern, "status_errors": int((got[3] != 0).sum()),
                     "parity": {"reads_checked": check, "mismatching_reads": len(bad)},
                     "tail_dp": {"cells_reference_would_compute": cells, "cells_planned": plan["cells"], "tiles": plan["trees"], "tails_aligned_in_place": plan["in_place"]}}
        dev.close(); index.close()
    return out


def secondary_seams(ordinal, n_problems=4000, check=40):
    """Secondary fields for the entry points outside the headline path: the chaining seams (seeds -> candidate transitions ->
    find_best_chains) and multi-mapping (max_multimaps = 3 on a repeat graph).  Kernel time only, with a parity count against
    the CPU restatement on a sample."""
    import helpers as H
    import test_chain_golden as TC
    import test_chain_candidates as TK
    from vg_b200 import capi, synth
    out = {}
    threads, _ = usable_cpus()
    g = synth.make_variant_graph()
    index = g.build_index()
    dev = capi.Device(index, ordinal)
    rng = np.random.default_rng(77)
    problems, anchors = [], []
    for _ in range(n_problems):
        h = int(rng.integers(0, len(g.hap_node)))
        base = int(rng.integers(0, len(g.hap_node[h]) - 1600))
        starts = sorted(set(int(x) for x in rng.integers(0, 1500, size=int(rng.integers(8, 64)))))
        jitter = rng.integers(-3, 4, size=len(starts))
        seeds = [(2 * int(g.hap_node[h][base + s]), int(g.hap_off[h][base + s])) for s in starts]
        A = np.zeros(len(starts), capi.chain_anchor_dt)
        A["read_start"] = np.maximum(0, np.asarray(starts) + jitter); A["length"] = 12; A["score"] = rng.integers(5, 13, size=len(starts))
        A["end_hint_offset"] = 12; A["base_seed_length"] = 12
        order = np.argsort(A["read_start"], kind="stable")
        problems.append([seeds[i] for i in order]); anchors.append(A[order])
    best_c = best_d = None
    for _ in range(2):
        cands = dev.chain_candidates_batch(problems, 300)
        best_c = dev.kernel_ms() if best_c is None else min(best_c, dev.kernel_ms())
        p = TC.params(max_chains=2)
        got = dev.chain_batch(list(zip(anchors, cands)), p)
        best_d = dev.kernel_ms() if best_d is None else min(best_d, dev.kernel_ms())
    bad = 0
    for i in range(check):
        want_c = TK.oracle_candidates(index, problems[i], 300)
        bad += int(cands[i].tobytes() != want_c.tobytes() or got[i] != TC.oracle_chain(anchors[i], want_c, p))
    out["chaining seams (gb_chain_candidates_batch + gb_chain_batch), config-2 graph"] = {
        "problems": n_problems, "seeds": int(sum(len(x) for x in problems)), "candidates": int(sum(len(c) for c in cands)),
        "candidates_kernel_ms": best_c, "chain_kernel_ms": best_d, "problems_per_s": n_problems / ((best_c + best_d) / 1e3),
        "parity": {"problems_checked": check, "mismatching_problems": bad}}
    dev.close(); index.close()

    g = synth.make_variant_graph(length=60000, n_snp=100, n_ins=10, n_del=10, n_haps=4, seed=23, repeat_unit=600, repeat_copies=6)
    index = g.build_index()
    dev = capi.Device(index, ordinal)
    n, k, chk = 100_000, 3, 5000
    rs = synth.simulate_reads(g, n, length=150, sub_rate=0.01, seed=36)
    p = H.default_map_params(); p.max_multimaps = k
    rbuf, qbuf, read_off = H.pack_reads(rs.reads, rs.quals)
    best = None
    for _ in range(2):
        got = dev.map_arrays(rbuf, qbuf, read_off, p)
        best = dev.kernel_ms() if best is None else min(best, dev.kernel_ms())
    want = H.oracle_map(index, rs.reads[:chk], rs.quals[:chk], p, threads=threads)
    sub = tuple(np.concatenate([got[0][j * n: j * n + chk] for j in range(k)]) if i == 0 else (got[i][:chk] if i == 3 else got[i]) for i in range(4))
    bad = H.compare_alignments(sub, want, chk, k=k)
    out["max_multimaps = 3, repeat graph (6 copies of a 600 bp unit), 150 bp SE"] = {
        "reads": n, "reads_per_s": n / (best / 1e3), "kernel_ms": best,
        "secondary_records": int(((got[0]["flags"] & capi.GB_ALN_SECONDARY) != 0).sum()),
        "parity": {"reads_checked": chk, "records_checked": chk * k, "mismatching_records": len(bad)}}
    dev.close(); index.close()
    return out


# ---------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads (not pairs) per GPU per step")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--rescue-attempts", type=int, default=15, help="MinimizerMapper::max_rescue_attempts (vg giraffe default 15)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --reads per GPU (configs[1]); strong: --total-reads split over the GPUs, identical total input for every N (configs[2])")
    ap.add_argument("--total-reads", type=int, default=100_000_000, help="strong scaling: reads of the whole job (BASELINE.json configs[2]: 100M)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (configs[3], configs[4], single-end) on rank 0 at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the alignment records the timed path returned in its last step (rank 0's reads; "
                         f"a fixed, seeded sample of {DUMP_READS} reads when there are more) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    # stdout carries exactly one line, the JSON: anything a library prints there (NCCL's version banner) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit_line(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_reads = args.reads - args.reads % 2
    BLOCK_PAIRS = 500_000                       # strong scaling: the job is a fixed sequence of seeded blocks, a rank takes a contiguous run
    if args.scaling == "strong":
        n_blocks = max(world, args.total_reads // (2 * BLOCK_PAIRS))
        from vg_b200 import shard as _sh
        blk_lo, blk_hi = _sh.shard_pairs(n_blocks, rank, world)
        n_reads = 2 * BLOCK_PAIRS * (blk_hi - blk_lo)

    import helpers as H

    if args.impl == "reference":
        # The reference arm: vg cannot be built here (all deps/ submodules are empty), so this times the
        # CPU restatement of the same path (oracle/) with every host thread, on rank 0 only.
        if rank != 0:
            return 0
        g, index = make_graph_and_index()
        params = H.paired_params(FRAG_MEAN, FRAG_SD)
        params.max_rescue_attempts = args.rescue_attempts
        lib, flags = oracle_library()
        threads, cpu_note = usable_cpus()
        sample = min(n_reads, 4_000_000)
        reads_np, quals_np = simulate_pairs_numpy(g, sample // 2, 22)
        rate, used, dt, _, threads = cpu_map_rate(index, reads_np, quals_np, params, threads, target_seconds=min(args.cpu_seconds, 10.0))
        out = H.oracle_out_buffers(used, params)
        times = []
        for s in range(args.warmup + args.steps):
            t = time.time()
            H.oracle_map_paired(index, reads_np[:used], quals_np[:used], params, threads=threads, out=out)
            if s >= args.warmup:
                times.append(time.time() - t)
        if args.dump_outputs:
            idx = dump_sample(used)
            aln_s = out[0][idx]
            dump_outputs(args.dump_outputs, idx, aln_s, out[3][idx], aln_s["mapping_off"], aln_s["edit_off"],
                         lambda i: out[1][i], lambda i: out[2][i])
        ms = 1e3 * float(np.mean(times))
        value = used / (ms / 1e3)
        line = {
            "impl": "reference", "metric": "giraffe reads/sec (150 bp PE, synthetic)", "value": value, "unit": "reads/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "mapper": f"map_paired, vg giraffe defaults (--rescue-attempts {args.rescue_attempts}), forced fragment distribution",
                       "reads_per_step": used, "sample": f"{used} reads of the same generator (error model, graph and seed family) per step: a bounded sample of the GPU arm's {n_reads}-read step",
                       "note": "CPU restatement of vg giraffe (oracle/, OpenMP over read pairs); vg itself cannot be built in this image"},
            "cpu_baseline": {"value": value, "unit": "reads/s", "cores": usable_cpus()[0], "threads": threads, "kind": "port", "sample": f"{used} reads per step, {threads} OpenMP threads, {flags}, {cpu_note}"},
            "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        emit_line(line)
        return 0

    import torch
    import torch.distributed as dist
    from vg_b200 import capi, shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)

    g, index = make_graph_and_index()
    dev = capi.Device(index, local_rank)
    lib = capi.load_library()
    params = H.paired_params(FRAG_MEAN, FRAG_SD)
    params.max_rescue_attempts = args.rescue_attempts
    stream = torch.cuda.Stream(device=device)          # the library's kernels and torch's events share this stream
    torch.cuda.set_stream(stream)
    lib.gb_device_set_stream(dev.handle, C.c_void_p(stream.cuda_stream))

    t = time.time()
    if args.scaling == "strong":
        d_reads = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, device=device)
        for bi in range(blk_lo, blk_hi):          # block bi is the same reads whatever the number of GPUs
            r_blk, _ = simulate_pairs_torch(g, BLOCK_PAIRS, 1000 + bi, device)
            d_reads[2 * BLOCK_PAIRS * (bi - blk_lo): 2 * BLOCK_PAIRS * (bi - blk_lo + 1)] = r_blk
        d_quals = torch.full_like(d_reads, 30)
    else:
        d_reads, d_quals = simulate_pairs_torch(g, n_reads // 2, 22 + rank, device)
    torch.cuda.synchronize()
    log(f"[bench] rank {rank}: {n_reads} reads generated on the GPU in {time.time() - t:.1f}s")
    d_read_off = (torch.arange(n_reads + 1, dtype=torch.int64, device=device) * READ_LEN)

    # ---- output buffers (device) ----
    MAP_PER, EDIT_PER = 14, 20
    d_aln = torch.zeros((n_reads, 32), dtype=torch.uint8, device=device)
    d_maps = torch.zeros((n_reads * MAP_PER, 8), dtype=torch.uint8, device=device)
    d_edits = torch.zeros((n_reads * EDIT_PER,), dtype=torch.int32, device=device)
    d_status = torch.zeros((n_reads,), dtype=torch.uint8, device=device)
    CHUNK = 1_000_000 if n_reads % 1_000_000 == 0 else 1 << 20     # equal launches, so the last chunk's stage timers are typical
    n_chunks = (n_reads + CHUNK - 1) // CHUNK
    d_totals = torch.zeros((n_chunks, 2), dtype=torch.int64, device=device)

    def device_step():
        """whole batch, device-resident, chunked to bound the intermediate pools"""
        for ci in range(n_chunks):
            c0 = ci * CHUNK
            cn = min(CHUNK, n_reads - c0)
            off = d_read_off[c0: c0 + cn + 1] - d_read_off[c0]
            rc = lib.gb_map_batch_device(dev.handle, C.byref(params), 1, cn,
                                         C.c_void_p(d_reads[c0].data_ptr()), C.c_void_p(d_quals[c0].data_ptr()),
                                         C.c_void_p(off.data_ptr()), READ_LEN,
                                         C.c_void_p(d_aln[c0].data_ptr()), C.c_void_p(d_maps[c0 * MAP_PER].data_ptr()), cn * MAP_PER,
                                         C.c_void_p(d_edits[c0 * EDIT_PER:].data_ptr()), cn * EDIT_PER,
                                         C.c_void_p(d_status[c0:].data_ptr()), C.c_void_p(d_totals[ci].data_ptr()))
            if rc != 0:
                raise capi.GbError(rc, "gb_map_batch_device")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed region 1: device-resident ----
    for _ in range(args.warmup):
        device_step()
    barrier()
    stage_ms = np.zeros(4)
    launches0 = dev.launches()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(stream)
    for _ in range(args.steps):
        device_step()
        # stage timers belong to the last chunk; scale by the chunk count for the share
    ev[1].record(stream)
    barrier()
    dev_ms = ev[0].elapsed_time(ev[1]) / args.steps
    clocks = sampler.stop()
    launches = (dev.launches() - launches0) // max(args.steps, 1)
    last_stage = np.array(dev.stage_times())
    kernel_times = dev.kernel_times()                  # every kernel of the last chunk, CUDA events between the launches
    plan_stats = dev.plan_stats()
    pool_overflow = dev.pool_overflow()                # the device entry cannot rerun a batch: an overflow would void the numbers
    if world > 1:
        tms = torch.tensor([dev_ms], device=device)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        dev_ms = float(tms.item())
    job_reads = 2 * BLOCK_PAIRS * n_blocks if args.scaling == "strong" else world * n_reads      # all ranks together
    value = job_reads / (dev_ms / 1e3)

    totals = d_totals.cpu().numpy()
    status_bad = int((d_status != 0).sum().item())
    aln_np = d_aln[: min(n_reads, 2_000_000)].cpu().numpy().view(capi.alignment_dt).reshape(-1)
    mapped_frac = float((aln_np["flags"] & 1).mean())
    mapq60 = float((aln_np["mapq"] == 60).mean())
    maps_per_read = float(totals[:, 0].sum()) / n_reads
    edits_per_read = float(totals[:, 1].sum()) / n_reads

    # ---- timed region 2: end to end through the host-buffer C-ABI (pinned host memory) ----
    h_reads = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, pin_memory=True)
    h_quals = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, pin_memory=True)
    h_reads.copy_(d_reads)
    h_quals.copy_(d_quals)
    torch.cuda.synchronize()
    h_off = torch.arange(n_reads + 1, dtype=torch.int64) * READ_LEN
    h_aln = torch.zeros((n_reads, 32), dtype=torch.uint8, pin_memory=True)
    h_maps = torch.zeros((n_reads * MAP_PER, 8), dtype=torch.uint8, pin_memory=True)
    h_edits = torch.zeros((n_reads * EDIT_PER,), dtype=torch.int32, pin_memory=True)
    h_status = torch.zeros((n_reads,), dtype=torch.uint8, pin_memory=True)
    used = (C.c_uint64(), C.c_uint64())

    def e2e_step():
        rc = lib.gb_map_paired_batch(dev.handle, C.byref(params), n_reads, C.c_void_p(h_reads.data_ptr()), C.c_void_p(h_quals.data_ptr()),
                                     C.c_void_p(h_off.data_ptr()), C.c_void_p(h_aln.data_ptr()), C.c_void_p(h_maps.data_ptr()),
                                     n_reads * MAP_PER, C.c_void_p(h_edits.data_ptr()), n_reads * EDIT_PER, C.c_void_p(h_status.data_ptr()),
                                     C.byref(used[0]), C.byref(used[1]))
        if rc != 0:
            raise capi.GbError(rc, "gb_map_paired_batch")

    # ---- multi-GPU emission: whole records (headers + mappings + edits) to rank 0 over NCCL / NVLink ----
    # The host-buffer call leaves its records in HBM too (output mirror); their gather runs on a side stream while the next
    # step maps, exact sizes, no padding, sizes exchanged on a host-side gloo group (no device sync); rank 0 lands every
    # rank's records in pinned host memory (what an AlignmentEmitter would consume).
    emit = None
    if world > 1:
        side = torch.cuda.Stream(device=device)
        gloo = dist.new_group(backend="gloo")
        m_aln = torch.zeros((n_reads, 32), dtype=torch.uint8, device=device)
        m_maps = torch.zeros((n_reads * MAP_PER, 8), dtype=torch.uint8, device=device)
        m_edits = torch.zeros((n_reads * EDIT_PER,), dtype=torch.int32, device=device)
        rcm = lib.gb_device_set_output_mirror(dev.handle, C.c_void_p(m_aln.data_ptr()), C.c_void_p(m_maps.data_ptr()), n_reads * MAP_PER,
                                              C.c_void_p(m_edits.data_ptr()), n_reads * EDIT_PER)
        assert rcm == 0
        caps = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(caps, torch.tensor([n_reads], dtype=torch.int64), group=gloo)
        recv = host_all = None
        if rank == 0:
            recv = [None if r == 0 else (torch.empty((int(c), 32), dtype=torch.uint8, device=device), torch.empty((int(c) * MAP_PER, 8), dtype=torch.uint8, device=device),
                                         torch.empty((int(c) * EDIT_PER,), dtype=torch.int32, device=device)) for r, c in enumerate(caps)]
            host_all = [None if r == 0 else (torch.empty((int(c), 32), dtype=torch.uint8, pin_memory=True), torch.empty((int(c) * MAP_PER, 8), dtype=torch.uint8, pin_memory=True),
                                             torch.empty((int(c) * EDIT_PER,), dtype=torch.int32, pin_memory=True)) for r, c in enumerate(caps)]
        emitted = {"records": 0, "mappings": 0}

        def emit():
            """gather of the step that just finished; returns immediately (work is queued on the side stream)"""
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                nm, ne = int(used[0].value), int(used[1].value)
                reqs, parts = shard.gather_records(m_aln, m_maps[:nm], m_edits[:ne], rank, world, counts_group=gloo, out=recv)
                for rq in reqs:
                    rq.wait()                      # stream-ordered for NCCL: the side stream waits, the host does not
                if rank == 0:
                    for r in range(1, world):
                        for src, dst in zip(parts[r], host_all[r]):
                            dst[: src.shape[0]].copy_(src, non_blocking=True)
                    emitted["records"] = sum(int(pt[0].shape[0]) for pt in parts)
                    emitted["mappings"] = sum(int(pt[1].shape[0]) for pt in parts)

    e2e_warm = min(args.warmup, 3)
    for _ in range(e2e_warm):
        e2e_step()
        if emit:
            emit()
    barrier()
    if emit:
        side.synchronize()
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t0 = time.time()
    ev2[0].record(stream)
    for _ in range(args.steps):
        if emit:
            side.synchronize()                     # the mirror is about to be overwritten: the previous step's gather must have left
        e2e_step()
        if emit:
            emit()
    if emit:
        stream.wait_stream(side)                   # the last gather is inside the timed region
    ev2[1].record(stream)
    barrier()
    if emit:
        side.synchronize()
    e2e_ms_dev = ev2[0].elapsed_time(ev2[1]) / args.steps
    e2e_ms_wall = 1e3 * (time.time() - t0) / args.steps
    e2e_ms = max(e2e_ms_dev, e2e_ms_wall)
    if world > 1:
        tms = torch.tensor([e2e_ms], device=device)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        e2e_ms = float(tms.item())
    e2e_value = job_reads / (e2e_ms / 1e3)
    h2d = 2 * n_reads * READ_LEN + 8 * (n_reads + 1)
    d2h = 32 * n_reads + n_reads + 8 * used[0].value + 4 * used[1].value

    # parity spot check of the e2e output against the device-resident output
    h_aln_np = h_aln.numpy().view(capi.alignment_dt).reshape(-1)
    same_scores = bool((h_aln_np["score"][: len(aln_np)] == aln_np["score"]).all())

    if args.dump_outputs and rank == 0:
        # the headline path's last timed step: gb_map_batch_device per chunk, whose read ids and pool offsets are
        # relative to the chunk's slice of the buffers
        idx = dump_sample(n_reads)
        d_idx = torch.from_numpy(idx).to(device)
        aln_s = d_aln[d_idx].cpu().numpy().view(capi.alignment_dt).reshape(-1)
        chunk0 = idx // CHUNK * CHUNK
        aln_s["read_id"] += chunk0.astype(np.uint32)
        dump_outputs(args.dump_outputs, idx, aln_s, d_status[d_idx].cpu().numpy(),
                     chunk0 * MAP_PER + aln_s["mapping_off"], chunk0 * EDIT_PER + aln_s["edit_off"],
                     lambda i: d_maps[torch.from_numpy(i).to(device)].cpu().numpy().view(capi.mapping_dt).reshape(-1),
                     lambda i: d_edits[torch.from_numpy(i).to(device)].cpu().numpy().view(np.uint32))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- CPU baseline on a bounded sample (rank 0) ----
    threads, cpu_note = usable_cpus()
    _, flags = oracle_library()
    sample_cap = min(n_reads, 6_000_000)
    reads_np = h_reads[:sample_cap].numpy()
    quals_np = h_quals[:sample_cap].numpy()
    cpu_rate, cpu_sample, cpu_dt, cpu_res, threads = cpu_map_rate(index, reads_np, quals_np, params, threads, target_seconds=args.cpu_seconds)
    counters = cpu_res[4]
    # parity of the timed GPU batch against the CPU run on the sample
    got = (h_aln_np[:cpu_sample], h_maps.numpy().view(capi.mapping_dt).reshape(-1), h_edits.numpy().view(np.uint32), h_status.numpy()[:cpu_sample])
    # first and last reads of the CPU sample: the sample spans several host chunks of the e2e call
    half = min(cpu_sample, 20000) // 2
    check_idx = list(range(half)) + list(range(cpu_sample - half, cpu_sample))
    check_n = len(check_idx)
    bad = H.compare_alignments(got, cpu_res, cpu_sample, indices=check_idx)

    B, terms, per_kernel = algorithmic_bytes_per_read(READ_LEN, counters, cpu_sample, maps_per_read, edits_per_read)
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    names = ["seed_kernel_pe", "extend_kernel", "align_kernel_pe", "compact"]
    # Per-kernel device times are measured live by the library (CUDA events between the launches of the last chunk,
    # gb_kernel_times); the dominant KERNEL is the longest of them.  Its algorithmic bytes are the term of B(read) its
    # stage touches (the align-stage kernels share one term: qualities, tail subgraphs, the output record).
    kdict = {}
    for kname, kms in kernel_times:
        kdict[kname] = kdict.get(kname, 0.0) + kms
    dom_name = max(kdict, key=kdict.get)
    term = "seed_kernel_pe" if dom_name.startswith("seed_kernel") else ("extend_kernel" if dom_name.startswith("extend") else ("compact" if dom_name.startswith("compact") else "align_kernel_pe"))
    chunk_reads = min(CHUNK, n_reads) if n_reads % CHUNK == 0 or n_reads < CHUNK else n_reads - (n_chunks - 1) * CHUNK
    dom_ms = float(kdict[dom_name])
    B_dom = float(per_kernel[term])
    achieved = B_dom * chunk_reads / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else None
    # dram__bytes_read.sum + dram__bytes_write.sum of that kernel's launch from the committed ncu --set full capture of THIS
    # command (profiles/ncu_summary_r02.json, keyed by kernel name and stamped with the commit it was taken at)
    traffic, traffic_commit = None, None
    try:
        prof = json.loads((ROOT / "profiles" / "ncu_summary_r02.json").read_text())
        full = prof["kernels"][dom_name]
        traffic = float(full["dram_bytes_per_launch"]) * chunk_reads / float(prof["reads_per_launch"])
        traffic_commit = prof.get("commit")
    except Exception:
        pass
    # The path is issue-bound, not HBM-bound (DESIGN.md §5): the second view of the same kernel is instruction issue — warp
    # instructions of one launch (from the same ncu capture) over the LIVE launch time, against SMs x 4 schedulers x the SM clock
    # sampled during the timed region.
    issue = None
    try:
        winst = float(prof["kernels"][dom_name]["ncu_full"]["warp_instructions"]) * chunk_reads / float(prof["reads_per_launch"])
        sms = torch.cuda.get_device_properties(device).multi_processor_count
        clock_hz = float(clocks["sm_mhz"]) * 1e6
        peak_i = sms * 4 * clock_hz
        issue = {"kernel": dom_name, "warp_instructions_per_launch": winst, "warp_instructions_per_read": winst / chunk_reads,
                 "achieved_warp_inst_per_s": winst / (dom_ms / 1e3), "peak_warp_inst_per_s": peak_i,
                 "frac": (winst / (dom_ms / 1e3)) / peak_i, "profile_commit": traffic_commit,
                 "note": "instruction counts from profiles/ncu_summary_r02.json, time and clock measured in this run"}
    except Exception:
        pass

    secondary = None
    if world == 1 and not args.no_secondary:
        dev.close()
        try:
            secondary = secondary_workloads(local_rank)
        except Exception as e:                       # never lose the headline line to a secondary workload
            secondary = {"error": repr(e)}
        try:
            secondary.update(secondary_seams(local_rank))
        except Exception as e:
            secondary["seams_error"] = repr(e)
    line = {
        "metric": "giraffe reads/sec (150 bp PE, synthetic)", "value": value, "unit": "reads/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {
            "workload": WORKLOAD,
            "reads_per_gpu_per_step": n_reads, "pairs_per_gpu_per_step": n_reads // 2,
            "total_reads_per_step": job_reads,
            "emission": (None if world == 1 else {"what": "whole records (32 B header + mappings + edits) of every rank gathered on rank 0 over NCCL, exact sizes, side stream overlapped with the next step, then to pinned host memory",
                                                   "records_on_rank0": emitted["records"], "mappings_on_rank0": emitted["mappings"]}),
            "mapper": f"map_paired, vg giraffe defaults (--rescue-attempts {args.rescue_attempts}), forced fragment distribution",
            "chunk_reads": CHUNK, "l2_policy": "inputs larger than L2 (3 GB of reads+qualities per step)",
            "mapped_fraction": mapped_frac, "mapq60_fraction": mapq60, "status_errors": status_bad,
            "parity_vs_cpu_sample": {"reads_checked": check_n, "mismatching_reads": len(bad)},
            "e2e_equals_device_scores": same_scores,
        },
        "clocks": clocks,
        "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms},
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_profile_commit": traffic_commit,
                     "issue": issue,
                     "kernel_ms_last_chunk": {k: round(v, 4) for k, v in kdict.items()},
                     "tail_plan": plan_stats, "pool_overflow": pool_overflow,
                     "algorithmic_bytes_per_read": B, "algorithmic_bytes_per_read_this_kernel": B_dom,
                     "per_kernel_bytes_per_read": {k: round(float(v), 1) for k, v in per_kernel.items()},
                     "terms": terms, "reads_per_launch": chunk_reads,
                     "launch_ms": dom_ms, "peak_source": peak_src,
                     "stage_ms_last_chunk": {n: float(x) for n, x in zip(names, last_stage)}},
        "cpu_baseline": {"value": cpu_rate, "unit": "reads/s", "cores": usable_cpus()[0], "threads": threads, "kind": "port",
                         "sample": f"{cpu_sample} reads ({cpu_sample // 2} pairs) of the same batch in {cpu_dt:.1f}s, oracle/ built {flags}, {threads} OpenMP threads over pairs, {cpu_note}"},
        "secondary": secondary,
    }
    emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
