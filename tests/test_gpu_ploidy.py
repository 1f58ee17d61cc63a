"""Polyploid runs on the GPU (--ploidy): the phased VCF is the haploid one with GT split over the haplotypes, each
haplotype's FASTA is the C oracle's walk of its records, genotypes match the host build of the rule, and the command
line writes, replays, chains and compresses the per-haplotype files."""
import ctypes as C
import gzip
import re
import shutil
import sys

import numpy as np
import pytest

from mutation_simulator_b200 import records as R
from tests.helpers import GOLDEN, MS_CASES, engine_for, load_case, load_muts, oracle_contig_from_recs, read_fasta_simple, vcf_body
from tests.test_chain_core import lift_check, parse_chains
from tests.test_genotype_core import core, core_masks  # noqa: F401  (fixture)
from tests.test_gpu_bgzf import REPO, _cli, _genome, _ngpu, _no_date, _sampled_engine, run_main
from tests.test_gpu_chain import SV_ARGS, _read, _vcf_snps

pytestmark = pytest.mark.gpu
GT = re.compile(rb"\tGT\t[01|]+\n")


def haploid_gt(body: bytes) -> bytes:
    return GT.sub(b"\tGT\t1\n", body)


def _c1_engine(seed=7):
    sys.path.insert(0, str(REPO))
    import bench
    from mutation_simulator_b200.engine import Engine
    wl = bench.WORKLOADS["c1"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(seed)
    return eng, lengths, names


def _golden_engine(case):
    d, contigs = load_case(case)
    eng, genome, goff, lens = engine_for(contigs)
    recs, lit = R.build_records(genome, goff, lens, load_muts(case))
    eng.load_records(recs, lit)
    return eng


# ---- the phased VCF is the haploid one ----------------------------------------------------------------------------------
@pytest.mark.parametrize("case", MS_CASES + ["c1"])
def test_union_is_the_haploid_vcf(case):
    eng = _c1_engine()[0] if case == "c1" else _golden_engine(case)
    eng.apply()
    haploid = eng.vcf()
    assert len(haploid) > 0
    for ploidy, f in ((2, 0.35), (3, 0.0), (8, 1.0)):
        eng.genotype_draw(11, ploidy, f)
        off = eng.vcf_phased()
        body = eng.download(7).tobytes()
        assert off[-1] == len(body) and haploid_gt(body) == haploid
        if f == 1.0:
            assert body == haploid.replace(b"\tGT\t1\n", b"\tGT\t" + b"|".join([b"1"] * ploidy) + b"\n")
        fo, vo, _, _ = eng.contig_layout()                           # per-contig slices line up with the haploid ones
        assert [haploid_gt(body[off[i]:off[i + 1]]) for i in range(len(off) - 1)] == \
               [haploid[vo[i]:vo[i + 1]] for i in range(len(vo) - 1)]
    eng.close()


def test_device_masks_equal_the_host_build(core):  # noqa: F811
    eng = _sampled_engine()
    recs = eng.records(True)
    lens = [len(c[2]) for c in _genome()]
    for ploidy, f in ((2, 0.35), (5, 0.5), (8, 0.0)):
        eng.genotype_draw(2024 + ploidy, ploidy, f)
        got = eng.genotypes()
        assert got.tobytes() == core_masks(core, recs, lens, 2024 + ploidy, ploidy, f).tobytes()
    eng.close()


# ---- each haplotype is its subset ----------------------------------------------------------------------------------------
def _haplotypes_match_oracle(eng, contigs, seed, ploidy):
    recs, lit, masks = eng.records(True), eng.literals(), eng.genotypes()
    lens = [len(c[2]) for c in contigs]
    goff = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    for h in range(1, ploidy + 1):
        sub = recs[(masks >> (h - 1) & 1).astype(bool)]
        sub = sub[sub["type"] != 255]
        eng.select_haplotype(h)
        eng.apply()
        image = eng.fasta()
        assert len(eng.records()) == len(sub)
        written = C.c_int64(0)
        want = b""
        for ci, (name, long_name, seq, bpl) in enumerate(contigs):
            mine = sub[sub["contig"] == ci]
            fa, _ = oracle_contig_from_recs(seq, name, long_name, bpl, mine, lit, int(goff[ci]), seed, ci, written)
            want += fa
        assert image == want, f"haplotype {h}"
    eng.select_haplotype(0)


@pytest.mark.parametrize("ploidy", [2, 3])
def test_each_haplotype_is_its_subset(ploidy):
    eng = _sampled_engine()
    eng.genotype_draw(5, ploidy, 0.35)
    _haplotypes_match_oracle(eng, _genome(), 99, ploidy)
    eng.close()


def test_each_haplotype_is_its_subset_on_c1():
    eng, lengths, names = _c1_engine()
    eng.genotype_draw(7, 2, 0.35)
    contigs = []
    goff = np.concatenate(([0], np.cumsum(lengths))).astype(np.int64)
    for i, L in enumerate(lengths):
        contigs.append((names[i], names[i], eng.read_genome(int(goff[i]), int(L)).tobytes(), 60))
    _haplotypes_match_oracle(eng, contigs, 7, 2)
    eng.close()


def test_select_zero_restores_the_full_table():
    eng = _sampled_engine()
    fasta, vcf, recs = eng.fasta(), eng.vcf(), eng.records(True)
    eng.genotype_draw(3, 3, 0.35)
    eng.select_haplotype(2)
    assert (eng.records(True)["out"] == 0).all()                       # like a loaded table until its apply
    eng.apply()
    assert eng.fasta() != fasta
    eng.select_haplotype(0)
    assert eng.records(True).tobytes() == recs.tobytes()
    eng.apply()
    assert eng.fasta() == fasta and eng.vcf() == vcf and eng.records(True).tobytes() == recs.tobytes()
    eng.close()


def test_hom_fraction_one_gives_the_haploid_genome_on_every_haplotype():
    eng = _sampled_engine()
    fasta = eng.fasta()
    eng.genotype_draw(3, 4, 1.0)
    for h in range(1, 5):
        eng.select_haplotype(h)
        eng.apply()
        assert eng.fasta() == fasta
    eng.close()


def test_state_and_argument_errors():
    from mutation_simulator_b200._lib import MS_ERR_ARG, MS_ERR_STATE, MutSimError
    eng = _sampled_engine()
    for call in (lambda: eng.select_haplotype(1), lambda: eng.vcf_phased()):
        with pytest.raises(MutSimError) as e:
            call()
        assert e.value.code == MS_ERR_STATE
    for call in (lambda: eng.genotype_draw(1, 1, 0.5), lambda: eng.genotype_draw(1, 9, 0.5),
                 lambda: eng.genotype_draw(1, 2, 1.5), lambda: eng.genotype_draw(1, 2, -0.1),
                 lambda: eng.genotype_load(np.zeros(3, np.uint8), 2)):
        with pytest.raises(MutSimError) as e:
            call()
        assert e.value.code == MS_ERR_ARG
    eng.genotype_draw(1, 2, 0.5)
    with pytest.raises(MutSimError) as e:
        eng.select_haplotype(3)
    assert e.value.code == MS_ERR_ARG
    bad = eng.genotypes().copy()
    bad[0] = 4
    with pytest.raises(MutSimError) as e:
        eng.genotype_load(bad, 2)
    assert e.value.code == MS_ERR_ARG
    eng.select_haplotype(1)
    eng.load_records(eng.records(True), eng.literals())                 # new records clear the masks
    for call in (lambda: eng.select_haplotype(1), lambda: eng.vcf_phased()):
        with pytest.raises(MutSimError) as e:
            call()
        assert e.value.code == MS_ERR_STATE
    eng.close()


def test_device_and_host_phased_parse_agree():
    eng = _sampled_engine()
    eng.genotype_draw(8, 3, 0.35)
    eng.vcf_phased()
    body = eng.download(7).tobytes()
    contigs = _genome()
    dev, _, goff, lens = engine_for(contigs)
    assert dev.load_vcf_phased(body, 3)
    assert not dev.load_vcf_phased(haploid_gt(body), 3)                 # a haploid GT under ploidy 3 is irregular
    _, _, hmasks = R.records_from_vcf(body, [c[0] for c in contigs], goff, lens, ploidy=3)
    assert dev.genotypes().tobytes() == hmasks.tobytes() and len(set(hmasks.tolist())) > 2
    dev.vcf_phased()
    assert dev.download(7).tobytes() == body                             # re-emitted byte for byte
    with pytest.raises(ValueError, match="ploidy 2"):
        R.records_from_vcf(body, [c[0] for c in contigs], goff, lens, ploidy=2)
    dev.close(); eng.close()


# ---- command line ---------------------------------------------------------------------------------------------------------
def _run(tmp_path, out, *extra, tail=SV_ARGS, seed="5"):
    run_main([tmp_path / "in.fa", "-o", tmp_path / out, "-q", "-w", "--seed", seed, *extra] + list(tail))


def test_ploidy_one_is_the_default_in_every_mode(tmp_path):
    shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
    shutil.copy(GOLDEN / "rmt_it" / "in.fa", tmp_path / "r.fa")
    shutil.copy(GOLDEN / "rmt_it" / "in.rmt", tmp_path / "r.rmt")
    for tag, extra in (("a", []), ("b", ["--ploidy", "1"])):
        _run(tmp_path, tag + "args", "--chain", *extra)
        run_main([tmp_path / "in.fa", "-o", tmp_path / (tag + "vcf"), "-q", "--chain", *extra, "vcf", tmp_path / "aargs_ms.vcf"])
        run_main([tmp_path / "r.fa", "-o", tmp_path / (tag + "rmt"), "-q", "-w", "--seed", "3", *extra, "rmt", tmp_path / "r.rmt"])
        run_main([tmp_path / "r.fa", "-o", tmp_path / (tag + "it"), "-q", "-w", "--seed", "3", *extra, "it", "0.004"])
    names = sorted(p.name[1:] for p in tmp_path.iterdir() if p.name.startswith("a") and "_ms" in p.name)
    assert names == sorted(p.name[1:] for p in tmp_path.iterdir() if p.name.startswith("b") and "_ms" in p.name)
    assert not any("_h1" in n for n in names)
    for n in names:
        a, b = (tmp_path / ("a" + n)).read_bytes(), (tmp_path / ("b" + n)).read_bytes()
        assert (_no_date(a) if n.endswith(".vcf") else a) == (_no_date(b) if n.endswith(".vcf") else b), n


def test_empty_contig_warning_with_and_without_ploidy(tmp_path, capsys):
    """Without -q / -w a contig that gets no mutation is reported on stderr, the same with no flag and --ploidy 1, and
    once per run with --ploidy 2."""
    rng = np.random.default_rng(4)
    seqs = [rng.choice(np.frombuffer(b"ACGT", np.uint8), n).tobytes() for n in (20_000, 10)]
    (tmp_path / "in.fa").write_bytes(b"".join(b">c%d\n" % i + s + b"\n" for i, s in enumerate(seqs)))
    err = {}
    for tag, extra in (("a", []), ("b", ["--ploidy", "1"]), ("c", ["--ploidy", "2"])):
        capsys.readouterr()
        run_main([tmp_path / "in.fa", "-o", tmp_path / tag, "--seed", "5", *extra, "args", "-sn", "0.01"])
        err[tag] = capsys.readouterr().err
    want = "No mutations could be generated on sequence 2 (mutation rates too low)"
    assert err["a"].count(want) == 1 and "sequence 1 " not in err["a"]
    assert err["b"] == err["a"] and err["c"] == err["a"]


@pytest.mark.parametrize("bgzip", [False, True])
def test_cli_round_trip_chain_and_bgzip(tmp_path, bgzip):
    z, gz = (["--bgzip"], ".gz") if bgzip else ([], "")
    shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
    _run(tmp_path, "h", "--ploidy", "2", "--chain")
    _run(tmp_path, "s", "--chain")                                                   # haploid, same seed
    assert not (tmp_path / "h_ms.fa").exists() and not (tmp_path / "h_ms.chain").exists()
    vcf = (tmp_path / "h_ms.vcf").read_bytes()
    assert haploid_gt(vcf_body(vcf)) == vcf_body((tmp_path / "s_ms.vcf").read_bytes())
    assert b"\tGT\t1|0\n" in vcf and b"\tGT\t0|1\n" in vcf
    ins = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / "in.fa")}
    for h in (1, 2):                                                                  # each chain lifts to its haplotype
        outs = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / f"h_ms_h{h}.fa")}
        snps = _vcf_snps(b"".join(l for l in vcf.splitlines(keepends=True)
                                  if l.startswith(b"#") or l.split(b"\t")[9][2 * (h - 1):2 * (h - 1) + 1] == b"1"))
        lift_check(parse_chains((tmp_path / f"h_ms_h{h}.chain").read_bytes()), ins, outs, snps, partition=False)
    if bgzip:
        _run(tmp_path, "z", "--ploidy", "2", "--chain", *z)
        for f in ("_ms.vcf", "_ms_h1.fa", "_ms_h2.fa", "_ms_h1.chain", "_ms_h2.chain"):
            a = gzip.decompress((tmp_path / f"z{f}.gz").read_bytes())
            b = (tmp_path / f"h{f}").read_bytes()
            assert (_no_date(a) if f.endswith(".vcf") else a) == (_no_date(b) if f.endswith(".vcf") else b), f
    # replay: the same haplotypes and phased body, device parse and host fallback (CRLF is declined by the device)
    run_main([tmp_path / "in.fa", "-o", tmp_path / "r", "-q", "--ploidy", "2", *z, "vcf", tmp_path / "h_ms.vcf"])
    (tmp_path / "crlf.vcf").write_bytes(vcf.replace(b"\n", b"\r\n"))
    run_main([tmp_path / "in.fa", "-o", tmp_path / "c", "-q", "--ploidy", "2", "vcf", tmp_path / "crlf.vcf"])
    for out, g in (("r", gz), ("c", "")):
        assert vcf_body(_read(tmp_path / f"{out}_ms.vcf{g}")) == vcf_body(vcf), out
        for h in (1, 2):
            a, b = _read(tmp_path / f"{out}_ms_h{h}.fa{g}"), (tmp_path / f"h_ms_h{h}.fa").read_bytes()
            assert a == b or a.replace(b"-", b"N") == b.replace(b"-", b"N"), (out, h)      # the Q6 '-' caveat of replays


def test_cli_replay_refuses_a_haploid_vcf(tmp_path):
    shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
    with pytest.raises(SystemExit):
        run_main([tmp_path / "in.fa", "-o", tmp_path / "r", "-q", "--ploidy", "2", "vcf", GOLDEN / "args_all" / "out.vcf"])


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_multi_gpu_ploidy_equals_single_gpu(tmp_path):
    from tests.test_gpu_multi import make_genome
    n = min(_ngpu(), 4)
    make_genome(tmp_path / "g.fa", [90_000, 70_011, 65_000, 40_000, 33_333, 20_000, 7, 1_000], 1)
    argv = ["-q", "--seed", "5", "--ploidy", "2", "--chain", "args", "-sn", "0.01", "-in", "0.002", "-de", "0.002", "-du",
            "0.002", "-iv", "0.002", "-tl", "0.002"]
    for d, k, env, port in (("a", 1, {}, 0), ("b", n, {}, 29663), ("c", n, {"MS_SHARD": "tiles"}, 29664)):
        (tmp_path / d).mkdir()
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "g")] + argv, k, port, **env)
    for f in ("g_ms.vcf", "g_ms_h1.fa", "g_ms_h2.fa", "g_ms_h1.chain", "g_ms_h2.chain"):
        want = (tmp_path / "a" / f).read_bytes()
        assert len(want) > 0
        for d in ("b", "c"):
            got = (tmp_path / d / f).read_bytes()
            assert (_no_date(got) if f.endswith(".vcf") else got) == (_no_date(want) if f.endswith(".vcf") else want), (d, f)
