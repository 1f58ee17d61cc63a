"""VCF replay parsed on the GPU (ms_load_vcf, Engine.load_vcf) and the `vcf` sub-command: the device parser gives the
host parser's record table, and replaying a run's own VCF rewrites that run's FASTA and VCF body byte for byte."""
import gzip
import shutil
import sys

import numpy as np
import pytest

from tests.helpers import GOLDEN, MS_CASES, engine_for, load_case, vcf_body
from tests.test_gpu_bgzf import REPO, _cli, _genome, _ngpu, _no_date, _sampled_engine, run_main
from tests.test_vcf_parse_core import random_genome, random_vcf

pytestmark = pytest.mark.gpu


def _host_engine(contigs, text, names, skip=False):
    from mutation_simulator_b200.records import records_from_vcf
    eng, _, goff, lens = engine_for(contigs)
    recs, lit = records_from_vcf(text, names, goff, lens, skip)
    eng.load_records(recs, lit)
    return eng


def assert_device_parse_equals_host(contigs, text, skip=False):
    names = [c[0] for c in contigs]
    dev, _, _, _ = engine_for(contigs)
    assert dev.load_vcf(text, skip)
    host = _host_engine(contigs, text, names, skip)
    assert dev.records(True).tobytes() == host.records(True).tobytes()      # before apply: out = 0
    assert dev.literals().tobytes() == host.literals().tobytes()
    assert dev.apply() == host.apply()
    assert dev.fasta() == host.fasta() and dev.vcf() == host.vcf()
    assert dev.records(True).tobytes() == host.records(True).tobytes()
    dev.close(); host.close()


@pytest.mark.parametrize("case", MS_CASES)
def test_golden_vcfs_load_like_the_host(case):
    d, contigs = load_case(case)
    assert_device_parse_equals_host(contigs, (d / "out.vcf").read_bytes())


@pytest.mark.parametrize("seed", range(6))
def test_random_vcfs_load_like_the_host(seed):
    rng = np.random.default_rng(seed)
    genome = random_genome(rng, iupac=seed % 2 == 0)
    contigs = [(n, n + b" desc", s, 60) for n, s in genome]
    text = random_vcf(rng, genome)
    assert_device_parse_equals_host(contigs, text)
    keep = sorted(rng.choice(len(contigs), 3, replace=False))       # one rank of a contig-sharded run
    assert_device_parse_equals_host([contigs[i] for i in keep], text, skip=True)


def test_a_sampled_runs_vcf_replays_to_its_outputs():
    eng = _sampled_engine()
    fasta, body = eng.fasta(), eng.vcf()
    eng.close()
    assert_device_parse_equals_host(_genome(), body)
    dev, _, _, _ = engine_for(_genome())
    assert dev.load_vcf(body)
    dev.apply()
    assert dev.fasta() == fasta and dev.vcf() == body
    dev.close()


def test_irregular_text_is_declined_and_overlaps_fail_like_the_host():
    from mutation_simulator_b200._lib import MutSimError
    d, contigs = load_case("args_all")
    text = (d / "out.vcf").read_bytes()
    eng, _, _, _ = engine_for(contigs)
    assert eng.load_vcf(text)
    n = len(eng.records(True))
    assert not eng.load_vcf(text.replace(b"\n", b"\r\n"))
    assert not eng.load_vcf(text.replace(b"\t.\tGT", b"\t.;X=1\tGT", 1))
    assert len(eng.records(True)) == n             # a declined text leaves the loaded table alone
    eng.close()
    name = contigs[0][0]
    bad = (name + b"\t5\t.\tA\tAC\t.\t.\tSVTYPE=INS;END=5;SVLEN=1\tGT\t1\n" + name + b"\t6\t.\tA\tG\t.\t.\t.\tGT\t1\n")
    errs = []
    for device in (True, False):
        eng, _, goff, lens = engine_for(contigs)
        with pytest.raises(MutSimError) as e:
            if device:
                eng.load_vcf(bad)
            else:
                from mutation_simulator_b200.records import records_from_vcf
                eng.load_records(*records_from_vcf(bad, [c[0] for c in contigs], goff, lens))
        errs.append(str(e.value))
        eng.close()
    assert errs[0] == errs[1] and "distinct positions" in errs[0]


def _setup(tmp_path, mode):
    if mode == "args":
        shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
        return ["args", "-sn", "0.01", "-in", "0.004", "-inmax", "9", "-de", "0.004", "-demax", "20", "-iv", "0.002",
                "-ivmax", "30", "-du", "0.002", "-dumax", "20", "-tl", "0.002", "-tlmax", "20"]
    shutil.copy(GOLDEN / "rmt_ranges" / "in.fa", tmp_path / "in.fa")
    shutil.copy(GOLDEN / "rmt_ranges" / "in.rmt", tmp_path / "in.rmt")
    return ["rmt", tmp_path / "in.rmt"]


def _read(p):
    b = p.read_bytes()
    return gzip.decompress(b) if p.suffix == ".gz" else b


@pytest.mark.parametrize("bgzip", [False, True])
@pytest.mark.parametrize("mode", ["args", "rmt"])
def test_cli_replay_of_a_runs_vcf_rewrites_its_outputs(tmp_path, mode, bgzip):
    tail = _setup(tmp_path, mode)
    z, gz = (["--bgzip"], ".gz") if bgzip else ([], "")
    run_main([tmp_path / "in.fa", "-o", tmp_path / "a", "-q", "-w", "--seed", "17"] + z + tail)
    run_main([tmp_path / "in.fa", "-o", tmp_path / "r", "-q"] + z + ["vcf", tmp_path / f"a_ms.vcf{gz}"])
    a_fa, r_fa = tmp_path / f"a_ms.fa{gz}", tmp_path / f"r_ms.fa{gz}"
    assert r_fa.read_bytes() == a_fa.read_bytes()
    body = vcf_body(_read(tmp_path / f"a_ms.vcf{gz}"))
    assert len(body) > 0 and vcf_body(_read(tmp_path / f"r_ms.vcf{gz}")) == body
    # a CRLF copy of the VCF takes the host parser and gives the same files
    (tmp_path / "crlf.vcf").write_bytes(_read(tmp_path / f"a_ms.vcf{gz}").replace(b"\n", b"\r\n"))
    run_main([tmp_path / "in.fa", "-o", tmp_path / "h", "-q"] + z + ["vcf", tmp_path / "crlf.vcf"])
    assert (tmp_path / f"h_ms.fa{gz}").read_bytes() == a_fa.read_bytes()
    assert vcf_body(_read(tmp_path / f"h_ms.vcf{gz}")) == body


@pytest.mark.parametrize("case", MS_CASES)
def test_cli_replay_of_the_reference_vcf(case, tmp_path):
    from tests.test_emu import assert_fasta_equal_up_to_silent_gap_snps
    d = GOLDEN / case
    shutil.copy(d / "in.fa", tmp_path / "in.fa")
    run_main([tmp_path / "in.fa", "-o", tmp_path / "r", "-q", "vcf", d / "out.vcf"])
    assert vcf_body((tmp_path / "r_ms.vcf").read_bytes()) == vcf_body((d / "out.vcf").read_bytes())
    assert_fasta_equal_up_to_silent_gap_snps((tmp_path / "r_ms.fa").read_bytes(), (d / "out.fa").read_bytes(), case)


def test_cli_errors_of_the_host_parser_and_the_same_file_guard(tmp_path, capsys):
    shutil.copy(GOLDEN / "tiny" / "in.fa", tmp_path / "in.fa")
    (tmp_path / "bad.vcf").write_bytes(b"##fileformat=VCFv4.3\nchr1\t3\t.\tA\n")
    with pytest.raises(SystemExit) as e:
        run_main([tmp_path / "in.fa", "-o", tmp_path / "r", "-q", "-c", "vcf", tmp_path / "bad.vcf"])
    assert e.value.code == 1
    assert capsys.readouterr().err.strip() == "ERROR: VCF line 2: expected at least 8 tab-separated fields"
    (tmp_path / "in_ms.vcf").write_bytes(b"x")
    with pytest.raises(SystemExit):
        run_main([tmp_path / "in.fa", "-o", tmp_path / "in", "-q", "-c", "vcf", tmp_path / "in_ms.vcf"])
    assert (tmp_path / "in_ms.vcf").read_bytes() == b"x" and not (tmp_path / "in_ms.fa").exists()


@pytest.mark.slow
def test_full_size_c2_shaped_replay():
    """GRCh38-shaped synthetic genome (3.1 Gbp, 24 contigs, bench.py's C2 mutation mix): replaying the run's own VCF
    body reproduces the FASTA image and the VCF body (device hashes)."""
    sys.path.insert(0, str(REPO))
    import bench
    from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF, Engine
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    fb, vb = eng.apply()
    want = eng.hash_ranges(BUF_FASTA, [0], [fb]), eng.hash_ranges(BUF_VCF, [0], [vb])
    body = eng.download(BUF_VCF)
    assert eng.load_vcf(body)
    assert eng.apply() == (fb, vb)
    assert np.array_equal(eng.hash_ranges(BUF_FASTA, [0], [fb]), want[0])
    assert np.array_equal(eng.hash_ranges(BUF_VCF, [0], [vb]), want[1])
    eng.close()


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_multi_gpu_vcf_mode_equals_single_gpu(tmp_path):
    from tests.test_gpu_multi import make_genome
    n = min(_ngpu(), 4)
    make_genome(tmp_path / "g.fa", [90_000, 70_011, 65_000, 40_000, 33_333, 20_000, 7, 1_000], 1)
    _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / "s"), "-q", "--seed", "5", "args", "-sn", "0.01", "-in", "0.002",
          "-de", "0.002", "-du", "0.001", "-iv", "0.001", "-tl", "0.002"], 1, 0)
    vcf = str(tmp_path / "s_ms.vcf")
    for d, k, env, port in (("a", 1, {}, 0), ("b", n, {}, 29643), ("c", n, {"MS_SHARD": "tiles"}, 29644)):
        (tmp_path / d).mkdir()
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "g"), "-q", "vcf", vcf], k, port, **env)
    a = {f: (tmp_path / "a" / f).read_bytes() for f in ("g_ms.fa", "g_ms.vcf")}
    assert a["g_ms.fa"] == (tmp_path / "s_ms.fa").read_bytes()
    for d in ("b", "c"):
        assert (tmp_path / d / "g_ms.fa").read_bytes() == a["g_ms.fa"], d
        assert _no_date((tmp_path / d / "g_ms.vcf").read_bytes()) == _no_date(a["g_ms.vcf"]), d
