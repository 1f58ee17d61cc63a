"""Paired-end reads on the GPU (--reads): device records equal the host build of the rule (ms_reads_core.h), the files
do not depend on the batch size, BGZF output inflates to the plain files, every read sits at its named coordinates of
the run's own FASTA, and runs with --reads write the same genome, VCF and chain files as runs without."""
import gzip
import shutil
import sys

import numpy as np
import pytest

from mutation_simulator_b200 import records as R
from mutation_simulator_b200.reads_writer import ReadsWriter, pair_counts, quality_char
from tests.helpers import GOLDEN, MS_CASES, engine_for, load_case, load_muts, read_fasta_simple
from tests.test_gpu_bgzf import REPO, _cli, _ngpu, _sampled_engine, run_main
from tests.test_gpu_chain import SV_ARGS
from tests.test_reads_core import COMP, core, parse_name, run_core  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def cfg(hap=1, L=50, M=200, S=30, E=0.01, seed=21):
    return dict(seed=seed, hap=hap, read_len=L, frag_mean=M, frag_sd=S, error_rate=E, qual=quality_char(E))


def device_vs_host(core, eng, g, n_pairs):  # noqa: F811
    """The device's records of all pairs equal the host build run on the engine's own FASTA image and records."""
    nb = eng.reads_write(g, n_pairs, 0, int(n_pairs.sum()))
    buf = eng.download(9).tobytes()
    assert len(buf) == 2 * nb
    img = eng.fasta()
    fo, _, _, _ = eng.contig_layout()
    all_recs = eng.records(include_dead=True)
    out_len = eng.contig_out_len()
    want1, want2 = [], []
    for c, n_c in enumerate(n_pairs):
        if not n_c:
            continue
        body_off = img.index(b"\n", int(fo[c])) + 1
        mseq = img[body_off:int(fo[c + 1])].replace(b"\n", b"")[:int(out_len[c])]
        a1, a2, _ = run_core(core, mseq, all_recs[all_recs["contig"] == c], eng.names[c], c, g["seed"], g["hap"], g["read_len"],
                             g["frag_mean"], g["frag_sd"], g["error_rate"], 0, int(n_c), bpl=int(eng._bpl[c]))
        want1.append(a1)
        want2.append(a2)
    assert buf[:nb] == b"".join(want1)
    assert buf[nb:] == b"".join(want2)
    sizes = eng.reads_size(g, n_pairs, 0, int(n_pairs.sum()))
    assert list(sizes) == [len(x) for x in _per_contig(want1, n_pairs)]
    return nb


def _per_contig(parts, n_pairs):
    it = iter(parts)
    return [next(it) if n else b"" for n in n_pairs]


def _golden_engine(case):
    d, contigs = load_case(case)
    eng, genome, goff, lens = engine_for(contigs)
    recs, lit = R.build_records(genome, goff, lens, load_muts(case))
    eng.load_records(recs, lit)
    return eng


@pytest.mark.parametrize("case", MS_CASES + ["sampled"])
def test_device_equals_host_core(core, case):  # noqa: F811
    eng = _sampled_engine() if case == "sampled" else _golden_engine(case)
    eng.apply()
    for hap, L, E in ((1, 50, 0.01), (2, 20, 0.2), (3, 1, 0.0)):
        n = pair_counts(2.0, eng.contig_out_len(), L, 3)
        g = cfg(hap=hap, L=L, M=max(L, 120), E=E)
        device_vs_host(core, eng, g, n)
        if n.sum() > 3:                                   # a range inside the table: the same records
            nb = eng.reads_write(g, n, 1, 2)
            full = eng.reads_write(g, n, 0, int(n.sum()))
            whole = eng.download(9).tobytes()
            eng.reads_write(g, n, 1, 2)
            part = eng.download(9).tobytes()
            recs1 = whole[:full].split(b"\n")
            assert part[:nb] == b"\n".join(recs1[4:12]) + b"\n"


@pytest.mark.parametrize("wl_name", ["c1", pytest.param("c2", marks=pytest.mark.slow)])
def test_device_equals_host_core_on_bench_workloads(core, wl_name):  # noqa: F811
    """C1, and the GRCh38-shaped C2 at low depth, haploid and the second haplotype of a diploid sample."""
    sys.path.insert(0, str(REPO))
    import bench
    from mutation_simulator_b200.engine import Engine
    wl = bench.WORKLOADS[wl_name]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(3)
    eng.genotype_draw(3, 2, 0.35)
    depth = 0.2 if wl_name == "c1" else 0.0005
    for hap in (0, 2):
        eng.select_haplotype(hap)
        eng.apply()
        n = pair_counts(depth, eng.contig_out_len(), 150, 1 if hap == 0 else 2)
        assert n.sum() > 100
        device_vs_host(core, eng, cfg(hap=max(hap, 1), L=150, M=500, S=50, E=0.001), n)


def test_write_after_size_reuses_its_draws(core):  # noqa: F811
    """ms_reads_write right after ms_reads_size of the same range and configuration formats that call's draws (fewer
    launches, the same bytes as the host build); another haplotype or range in between makes it draw again."""
    eng = _sampled_engine()
    eng.apply()
    n = pair_counts(1.0, eng.contig_out_len(), 60, 1)
    total = int(n.sum())
    g = cfg(L=60, M=200)

    def launches(f, *a):
        before = eng.stats()["kernel_launches"]
        r = f(*a)
        return r, eng.stats()["kernel_launches"] - before

    def fresh(g2, first, count):
        eng.load_records(eng.records(True), eng.literals())         # forget every sized range
        eng.apply()
        nb = eng.reads_write(g2, n, first, count)
        return eng.download(9).tobytes()[:2 * nb]

    want = {(h, f, c): fresh(cfg(hap=h, L=60, M=200), f, c) for h, f, c in ((1, 0, total), (2, 0, total), (1, 1, 3))}
    _, cold = launches(eng.reads_write, g, n, 0, total)
    eng.reads_size(g, n, 0, total)
    nb, warm = launches(eng.reads_write, g, n, 0, total)
    assert warm < cold
    assert eng.download(9).tobytes() == want[(1, 0, total)]
    eng.reads_size(g, n, 0, total)
    device_vs_host(core, eng, g, n)                                    # its first call is the reusing write
    for h, f, c in ((2, 0, total), (1, 1, 3)):                         # another haplotype, another range
        eng.reads_size(g, n, 0, total)
        nb, relaunch = launches(eng.reads_write, cfg(hap=h, L=60, M=200), n, f, c)
        assert relaunch > warm and eng.download(9).tobytes() == want[(h, f, c)], (h, f, c)
    assert want[(1, 0, total)] != want[(2, 0, total)]


def test_partitioned_writer_on_one_gpu(tmp_path):
    """The several-GPU writer with one rank: contig slices, and each contig cut in two slots as tile mode does, give
    the files of the one-GPU writer, plain and BGZF."""
    eng = _sampled_engine()
    eng.apply()
    g = cfg(L=100, M=300)
    n = pair_counts(2.0, eng.contig_out_len(), 100, 2)
    for bgzip in (False, True):
        want = _write(eng, g, n, tmp_path, f"w{bgzip:d}", 4 << 30, bgzip)
        for tag, slices, n_slots in (("ctg", [(c, c, 0, int(n[c])) for c in range(len(n))], len(n)),
                                     ("cut", [(2 * c + r, c, int(n[c]) * r // 2, int(n[c]) * (r + 1) // 2)
                                              for c in range(len(n)) for r in (0, 1)], 2 * len(n))):
            paths = [tmp_path / f"{tag}{bgzip:d}_R1.fq", tmp_path / f"{tag}{bgzip:d}_R2.fq"]
            w = ReadsWriter(paths, bgzip, 3000, create=False)
            w.write_partitioned(eng, g, n, slices, n_slots)
            w.write_partitioned(eng, dict(g, hap=2), n, slices, n_slots)
            w.close()
            got = [p.read_bytes() for p in paths]
            assert (got if not bgzip else [gzip.decompress(x) for x in got]) == \
                (want if not bgzip else [gzip.decompress(x) for x in want]), (tag, bgzip)


def _write(eng, g, n, tmp_path, tag, budget, bgzip=False):
    paths = [tmp_path / f"{tag}_R1.fq", tmp_path / f"{tag}_R2.fq"]
    w = ReadsWriter(paths, bgzip, budget)
    w.write(eng, g, n)
    w.write(eng, dict(g, hap=2), n)                     # a second haplotype continues both files
    w.close()
    return [p.read_bytes() for p in paths]


def test_batch_budget_does_not_change_the_files(tmp_path):
    from mutation_simulator_b200.bgzf import EOF
    eng = _sampled_engine()
    eng.apply()
    g = cfg(L=100, M=300)
    n = pair_counts(1.0, eng.contig_out_len(), 100, 2)
    want = _write(eng, g, n, tmp_path, "d", 4 << 30)
    assert len(want[0]) == len(want[1]) > 0
    for tag, budget in (("one", 1), ("kib", 3000)):
        assert _write(eng, g, n, tmp_path, tag, budget) == want, tag
    for tag, budget in (("zd", 4 << 30), ("z1", 1), ("zk", 5000)):
        z = _write(eng, g, n, tmp_path, tag, budget, bgzip=True)
        for zz, plain in zip(z, want):
            assert zz.endswith(EOF)
            assert gzip.decompress(zz) == plain, tag


def test_state_and_argument_errors():
    from mutation_simulator_b200._lib import MS_ERR_ARG, MS_ERR_STATE, MutSimError
    from tests.test_gpu_bgzf import _genome
    eng = engine_for(_genome())[0]
    g = cfg()
    n = np.ones(eng.n_contigs, np.int64)
    n[eng.contig_out_len() < 50] = 0

    def code(f, *a):
        with pytest.raises(MutSimError) as e:
            f(*a)
        return e.value.code

    assert code(eng.reads_size, g, n, 0, 1) == MS_ERR_STATE           # before an apply
    eng.load_records(np.zeros(0, R.REC_DTYPE))
    assert code(eng.reads_size, g, n, 0, 1) == MS_ERR_STATE           # records without an apply
    eng.apply_window(0, 2)
    assert code(eng.reads_write, g, n, 0, 1) == MS_ERR_STATE          # a window leaves buffer 0 partly valid
    eng.apply()
    assert eng.reads_write(g, n, 0, int(n.sum())) > 0
    for bad in (dict(hap=0), dict(hap=9), dict(read_len=0), dict(read_len=1001), dict(frag_mean=49), dict(frag_mean=10 ** 6 + 1),
                dict(frag_sd=-1), dict(frag_sd=100_001), dict(error_rate=1.0), dict(error_rate=-0.1), dict(qual=20)):
        assert code(eng.reads_size, dict(g, **bad), n, 0, 1) == MS_ERR_ARG, bad
    assert code(eng.reads_write, g, n, 0, int(n.sum()) + 1) == MS_ERR_ARG
    assert code(eng.reads_write, g, n, -1, 1) == MS_ERR_ARG
    neg = n.copy(); neg[0] = -1
    assert code(eng.reads_size, g, neg, 0, 0) == MS_ERR_ARG
    short = np.ones(eng.n_contigs, np.int64)
    assert code(eng.reads_size, g, short, 0, 1) == MS_ERR_ARG          # pairs on a contig shorter than the reads
    eng.adopt_output()
    assert code(eng.reads_write, g, n, 0, 1) == MS_ERR_STATE
    eng.apply()
    eng.reads_write(g, n, 0, 1)
    eng.load_records(np.zeros(0, R.REC_DTYPE))
    assert code(eng.reads_write, g, n, 0, 1) == MS_ERR_STATE          # new records


# ---- command line -------------------------------------------------------------------------------------------------------
READS = ["--reads", "3", "--read-length", "40", "--fragment-mean", "120", "--fragment-sd", "20", "--read-error-rate", "0"]


def check_reads_against_fasta(r1: bytes, r2: bytes, fastas, ploidy, L=40, depth=3.0):
    """Every read equals its haplotype's mutated contig at its named coordinates (E = 0), and each contig has the pairs
    the count rule gives."""
    seqs = [{c[0]: c[2] for c in read_fasta_simple(f)} for f in fastas]
    counts = {}
    for text, mate in ((r1, 1), (r2, 2)):
        lines = text.split(b"\n")
        assert lines[-1] == b"" and len(lines) % 4 == 1
        for k in range(0, len(lines) - 1, 4):
            nm, h, i, s, f, strand, _, _ = parse_name(lines[k])
            fwd = (mate == 1) == (strand == b"+")
            m = seqs[h - 1][nm]
            x = s if fwd else s + f - L
            assert lines[k + 1] == (m[x:x + L] if fwd else m[x:x + L][::-1].translate(COMP))
            assert lines[k + 2] == b"+" and lines[k + 3] == b"J" * L
            counts[(h, nm)] = counts.get((h, nm), 0) + (mate == 1)
    for h, s in enumerate(seqs, 1):
        for nm, m in s.items():
            assert counts.get((h, nm), 0) == pair_counts(depth, [len(m)], L, ploidy)[0], (h, nm)


def _outputs(tmp_path, prefix, ploidy, gz=""):
    names = [f"{prefix}_ms.vcf{gz}"] + ([f"{prefix}_ms_h{h}.fa{gz}" for h in range(1, ploidy + 1)] if ploidy > 1 else [f"{prefix}_ms.fa{gz}"])
    chains = [f"{prefix}_ms_h{h}.chain{gz}" for h in range(1, ploidy + 1)] if ploidy > 1 else [f"{prefix}_ms.chain{gz}"]
    return {n.replace(prefix, "", 1): (tmp_path / n).read_bytes() for n in names + chains}


@pytest.mark.parametrize("mode", ["args", "rmt"])
@pytest.mark.parametrize("ploidy", [1, 2])
def test_cli_round_trip_and_replay(tmp_path, mode, ploidy):
    if mode == "args":
        shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
        tail = SV_ARGS
    else:
        shutil.copy(GOLDEN / "rmt_ranges" / "in.fa", tmp_path / "in.fa")
        shutil.copy(GOLDEN / "rmt_ranges" / "in.rmt", tmp_path / "in.rmt")
        tail = ["rmt", tmp_path / "in.rmt"]
    common = [tmp_path / "in.fa", "-q", "-w", "--seed", "4", "--chain", "--ploidy", str(ploidy)]
    run_main(common + ["-o", tmp_path / "a"] + READS + tail)
    run_main(common + ["-o", tmp_path / "b"] + tail)
    assert _outputs(tmp_path, "a", ploidy) == _outputs(tmp_path, "b", ploidy)      # --reads changes no other file
    assert not (tmp_path / "b_ms_R1.fq").exists()
    fastas = [tmp_path / f"a_ms_h{h}.fa" for h in range(1, ploidy + 1)] if ploidy > 1 else [tmp_path / "a_ms.fa"]
    r1, r2 = (tmp_path / "a_ms_R1.fq").read_bytes(), (tmp_path / "a_ms_R2.fq").read_bytes()
    assert len(r1) == len(r2) > 0
    check_reads_against_fasta(r1, r2, fastas, ploidy)
    # replay of the run's VCF: the same genome, so the same pairs; the lifts follow the replayed table, whose records
    # may differ from the run's (a deletion replays with its anchor base), so only the names' lifts may differ
    run_main([tmp_path / "in.fa", "-q", "-w", "--seed", "4", "--ploidy", str(ploidy), "-o", tmp_path / "v"] + READS +
             ["vcf", tmp_path / "a_ms.vcf"])
    v1, v2 = (tmp_path / "v_ms_R1.fq").read_bytes(), (tmp_path / "v_ms_R2.fq").read_bytes()
    check_reads_against_fasta(v1, v2, fastas, ploidy)
    strip = lambda t: [ln.rsplit(b":", 2)[0] if k % 4 == 0 else ln for k, ln in enumerate(t.split(b"\n"))]
    assert strip(v1) == strip(r1) and strip(v2) == strip(r2)
    # --bgzip: the same reads, compressed
    run_main(common + ["-o", tmp_path / "z", "--bgzip"] + READS + tail)
    assert gzip.decompress((tmp_path / "z_ms_R1.fq.gz").read_bytes()) == r1
    assert gzip.decompress((tmp_path / "z_ms_R2.fq.gz").read_bytes()) == r2


def test_cli_warns_once_for_contigs_without_pairs(tmp_path, capfd):
    rng = np.random.default_rng(5)
    with open(tmp_path / "in.fa", "wb") as fh:
        for i, n in enumerate((30, 2000, 50, 500)):          # two contigs shorter than one read
            fh.write(b">c%d\n" % i + rng.choice(list(b"ACGT"), n).astype(np.uint8).tobytes() + b"\n")
    argv = ["--seed", "4", "--ploidy", "2", "--reads", "4", "--read-length", "100", "--fragment-mean", "150"] + SV_ARGS
    run_main([tmp_path / "in.fa", "-o", tmp_path / "a"] + argv)
    err = capfd.readouterr().err
    out = [{c[0]: len(c[2]) for c in read_fasta_simple(tmp_path / f"a_ms_h{h}.fa")} for h in (1, 2)]
    none = [nm for nm in out[0] if out[0][nm] < 100 and out[1][nm] < 100]
    assert len(none) == 2 and err.count("No reads could be simulated") == 2
    assert "sequence 1 " in err and "sequence 3 " in err
    run_main([tmp_path / "in.fa", "-o", tmp_path / "b", "-w"] + argv)
    assert "No reads" not in capfd.readouterr().err


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_multi_gpu_reads_equal_single_gpu(tmp_path):
    from tests.test_gpu_multi import make_genome
    n = min(_ngpu(), 4)
    make_genome(tmp_path / "g.fa", [90_000, 70_011, 65_000, 40_000, 33_333, 20_000, 7, 1_000], 1)
    argv = ["-q", "--seed", "5", "--reads", "2", "--read-length", "60", "--fragment-mean", "200", "args", "-sn", "0.01", "-in",
            "0.002", "-de", "0.002", "-du", "0.002", "-iv", "0.002", "-tl", "0.002"]
    for d, k, env, port in (("a", 1, {}, 0), ("b", n, {}, 29663), ("c", n, {"MS_SHARD": "tiles"}, 29664)):
        (tmp_path / d).mkdir()
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "g")] + argv, k, port, **env)
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "p"), "--ploidy", "2"] + argv, k, port + 20 if port else 0, **env)
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "z"), "--bgzip"] + argv, k, port + 10 if port else 0, **env)
    for f in ("g_ms_R1.fq", "g_ms_R2.fq", "p_ms_R1.fq", "p_ms_R2.fq"):
        want = (tmp_path / "a" / f).read_bytes()
        assert len(want) > 0
        for d in ("b", "c"):
            assert (tmp_path / d / f).read_bytes() == want, (d, f)
    for d in ("b", "c"):
        assert gzip.decompress((tmp_path / d / "z_ms_R1.fq.gz").read_bytes()) == (tmp_path / "a" / "g_ms_R1.fq").read_bytes()
