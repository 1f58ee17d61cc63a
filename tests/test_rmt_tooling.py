"""SURVEY.md §8 f4: the GFF -> RMT helper and the annotation-derived RMTs it produces (overlapping blocked ranges)."""
import re

import numpy as np
import pytest

from mutation_simulator_b200 import SimulationSettings, plan
from mutation_simulator_b200.fasta import FastaRecord
from mutation_simulator_b200.tools import gff_genes_2_rmt

GFF = """##gff-version 3
chr2\tsrc\tgene\t500\t900\t.\t+\t.\tID=g1
chr2\tsrc\tmRNA\t500\t900\t.\t+\t.\tID=t1
chr1\tsrc\tGene\t100\t400\t.\t-\t.\tID=g2
chr1\tsrc\tgene\t350\t800\t.\t+\t.\tID=g3
chr1\tsrc\tgene\t360\t370\t.\t+\t.\tID=g4
# comment
chr2\tsrc\tgene\t10\t20\t.\t+\t.\tID=g5
"""


class LengthsOnly:
    """The part of the Fasta surface SimulationSettings reads: names and lengths."""
    def __init__(self, lens):
        self.names = [f"c{i}" for i in range(len(lens))]
        self.lengths = np.array(lens, np.int64)
        self._r = [FastaRecord(n, n, None, 60, length=int(l)) for n, l in zip(self.names, lens)]

    def __getitem__(self, k):
        return self._r[k] if isinstance(k, (int, np.integer)) else self._r[self.names.index(k)]

    def keys(self):
        return self.names

    def __len__(self):
        return len(self.names)


def test_gff_helper_writes_what_the_reference_script_writes(tmp_path):
    (tmp_path / "a.gff3").write_text(GFF)
    assert gff_genes_2_rmt.main([str(tmp_path / "a.gff3"), "0.01"]) == 0
    got = (tmp_path / "a.rmt").read_text()
    # what the reference's data/scripts/gff_genes_2_rmt.py writes for GFF
    assert got == ("std\nit None\nsn 0.01\n\nchr 1 #chr2\n500-900 None\n10-20 None\n"
                   "chr 2 #chr1\n100-400 None\n350-800 None\n360-370 None\n")
    assert gff_genes_2_rmt.main([str(tmp_path / "a.gff3")]) == 1
    assert gff_genes_2_rmt.main([str(tmp_path / "nope.gff3"), "0.1"]) == 1
    assert gff_genes_2_rmt.main([str(tmp_path / "a.gff3"), "x"]) == 1


def test_overlapping_blocked_ranges_are_planned_as_their_union(tmp_path):
    """Gene intervals overlap and nest; the reference's gap filler then makes negative-length ranges and dies in
    random.sample.  The planner lets blocked ranges win: candidates only where no None range reaches."""
    (tmp_path / "a.gff3").write_text(GFF)
    gff_genes_2_rmt.main([str(tmp_path / "a.gff3"), "0.01"])
    fa = LengthsOnly([2000, 3000])
    sim = SimulationSettings.from_rmt(tmp_path / "a.rmt", fa, True)
    arr, n = plan.build_ranges(sim, fa.lengths)
    rows = [(arr[i].contig, arr[i].start, arr[i].stop, arr[i].limit) for i in range(n)]
    # chr 1: blocked 10-20, 500-900 (1-based)   chr 2: blocked 100-800 (union of 100-400, 350-800, 360-370)
    # (the head fillers 1-9 and 1-99 get int(len * 0.01) = 0 candidates and are dropped)
    assert rows == [(0, 20, 498, 499), (0, 900, 1999, 2000), (1, 800, 2999, 3000)]
    for i in range(n):
        assert arr[i].k == int(((arr[i].stop - arr[i].start) + 1) * 0.01)


# name: (sequences, genes per sequence, sequence length, longest gene)
ANNOTATIONS = {
    "one_chromosome": (1, 3000, 120_000_000, 100_000),
    "five_chromosomes": (5, 1000, 30_000_000, 100_000),
    "twenty_five_chromosomes": (25, 200, 20_000_000, 100_000),
    "dense_nested_genes": (3, 2500, 6_000_000, 5_000),
    "many_scaffolds": (400, 5, 500_000, 50_000),
}


def annotation_gff(n_seq, genes, seq_len, longest, seed):
    """A seeded genome annotation in GFF3: per sequence, genes of 200 bp to `longest` (log-uniform) at random places,
    sorted by start as annotation files are, so that they overlap and nest like real genes; every gene carries an mRNA
    and an exon, which the helper skips."""
    rng = np.random.default_rng(seed)
    out = ["##gff-version 3"]
    for s in range(n_seq):
        seqid = f"seq{s + 1}"
        out.append(f"##sequence-region {seqid} 1 {seq_len}")
        lens = np.exp(rng.uniform(np.log(200), np.log(longest), genes)).astype(np.int64)
        starts = rng.integers(1, seq_len - lens + 1)
        for g, i in enumerate(np.argsort(starts, kind="stable")):
            a, b = int(starts[i]), int(starts[i] + lens[i] - 1)
            strand = "+-"[g % 2]
            out.append(f"{seqid}\tsynthetic\tgene\t{a}\t{b}\t.\t{strand}\t.\tID=g{s}_{g}")
            out.append(f"{seqid}\tsynthetic\tmRNA\t{a}\t{b}\t.\t{strand}\t.\tID=t{s}_{g};Parent=g{s}_{g}")
            out.append(f"{seqid}\tsynthetic\texon\t{a}\t{min(b, a + 150)}\t.\t{strand}\t.\tParent=t{s}_{g}")
    return "\n".join(out) + "\n"


@pytest.mark.parametrize("name", sorted(ANNOTATIONS))
def test_annotation_rmts_parse_and_plan(name, tmp_path):
    """RMTs the GFF helper makes from whole-genome annotations: thousands of overlapping and nested None ranges over
    many sequences parse, and plan into sorted, in-bounds ranges that never touch a blocked interval."""
    gff = tmp_path / f"{name}.gff3"
    gff.write_text(annotation_gff(*ANNOTATIONS[name], seed=1))
    assert gff_genes_2_rmt.main([str(gff), "0.01"]) == 0
    p = gff.with_suffix(".rmt")
    ends, cur = {}, None
    for line in p.read_text().splitlines():
        m = re.match(r"chr (\d+)", line)
        if m:
            cur = int(m.group(1)); ends.setdefault(cur, 1000); continue
        m = re.match(r"(\d+)-(\d+)", line)
        if m and cur:
            ends[cur] = max(ends[cur], int(m.group(2)) + 1000)
    fa = LengthsOnly([ends.get(i + 1, 1000) for i in range(max(ends))])
    sim = SimulationSettings.from_rmt(p, fa, True)
    arr, n = plan.build_ranges(sim, fa.lengths)
    assert n > 1000
    blocked = {}
    for c in sim.chromosomes:
        blocked[c.number] = sorted((r.start, r.stop) for r in c.range_definitions if not r.mutation_settings.has_mutations)
    prev = (-1, -1)
    for i in range(n):
        a = arr[i]
        assert a.start <= a.stop < fa.lengths[a.contig] and a.limit <= fa.lengths[a.contig]
        assert (a.contig, a.start) > prev
        prev = (a.contig, a.stop)
    # no planned range touches a blocked interval
    for i in range(0, n, 97):
        a = arr[i]
        assert not any(s <= a.stop and e >= a.start for s, e in blocked[a.contig])
