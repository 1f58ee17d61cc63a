"""The chain file on the GPU (ms_chain_count / ms_chain_write, Engine.chain_*, ``--chain``): the device's bytes are the
format's restatement, every block names the same bases in the input and the mutated FASTA, and the CLI writes the
file in every mode, with and without --bgzip, on one GPU and on several."""
import gzip
import shutil
import sys

import numpy as np
import pytest

from mutation_simulator_b200 import records as R
from mutation_simulator_b200.chain_writer import first_ids
from tests.helpers import GOLDEN, MS_CASES, engine_for, read_fasta_simple
from tests.test_chain_core import core, golden_table, lift_check, parse_chains, random_table, restate, run_core  # noqa: F401
from tests.test_gpu_bgzf import REPO, _cli, _ngpu, run_main

pytestmark = pytest.mark.gpu


def device_chain(eng):
    from mutation_simulator_b200.engine import BUF_CHAIN
    n = eng.chain_count()
    off = eng.chain_write(first_ids(n))
    return eng.download(BUF_CHAIN).tobytes(), n, off


def _engine_with(recs, lens, names, rng=None):
    rng = rng or np.random.default_rng(0)
    seqs = [rng.choice(np.frombuffer(b"ACGTN", np.uint8), L).tobytes() for L in lens]
    eng, _, _, _ = engine_for([(n, n + b" x", s, 60) for n, s in zip(names, seqs)])
    eng.load_records(recs)
    eng.apply()
    return eng


@pytest.mark.parametrize("case", MS_CASES)
def test_device_equals_restatement_on_goldens(case):
    from tests.helpers import load_muts
    _, lens, names = golden_table(case)
    contigs = read_fasta_simple(GOLDEN / case / "in.fa")
    eng, genome, goff, _ = engine_for(contigs)
    recs, lit = R.build_records(genome, goff, lens, load_muts(case))
    eng.load_records(recs, lit)
    eng.apply()
    text, n, off = device_chain(eng)
    assert text == restate(recs, lens, names)
    assert int(off[-1]) == len(text) and int(n.sum()) == len(parse_chains(text))
    eng.close()


@pytest.mark.parametrize("seed", range(8))
def test_device_equals_restatement_on_random_tables(seed):
    rng = np.random.default_rng(seed)
    recs, lens, names = random_table(rng)
    eng = _engine_with(recs, lens, names, rng)
    text, n, _ = device_chain(eng)
    assert text == restate(recs, lens, names)
    start = 1 + int(rng.integers(0, 1 << 30))
    from mutation_simulator_b200.engine import BUF_CHAIN
    eng.chain_write(first_ids(n, start))
    assert eng.download(BUF_CHAIN).tobytes() == restate(recs, lens, names, start)
    eng.close()


@pytest.mark.parametrize("wl_name", ["c1", pytest.param("c2", marks=pytest.mark.slow)])
def test_device_equals_host_build_on_bench_workloads(core, wl_name):  # noqa: F811
    """C1, and C2 in full (GRCh38-shaped, 24 contigs): device bytes equal the host build of the emitter run on the
    downloaded record table."""
    sys.path.insert(0, str(REPO))
    import bench
    from mutation_simulator_b200.engine import Engine
    wl = bench.WORKLOADS[wl_name]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    eng.apply()
    text, n, off = device_chain(eng)
    want, wn, woff = run_core(core, eng.records(True), lengths, names)
    assert np.array_equal(n, wn) and np.array_equal(off, woff)
    assert text == want
    eng.close()


def test_state_and_source_errors():
    from mutation_simulator_b200._lib import MS_ERR_ARG, MS_ERR_STATE, MutSimError
    lens, names = [100, 100], [b"a", b"b"]
    rng = np.random.default_rng(1)
    seqs = [rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes() for L in lens]
    eng, _, _, _ = engine_for([(n, n, s, 60) for n, s in zip(names, seqs)])
    with pytest.raises(MutSimError) as e:
        eng.chain_count()
    assert e.value.code == MS_ERR_STATE
    recs = np.zeros(1, dtype=R.REC_DTYPE)
    recs[0] = (10, 0, 5, 0, 150, R.K_RAW, R.T_DU, 0, 0, 0)       # copies from contig b into contig a
    eng.load_records(recs)
    with pytest.raises(MutSimError) as e:
        eng.chain_count()
    assert e.value.code == MS_ERR_STATE                          # loaded, not applied
    eng.apply()
    with pytest.raises(MutSimError) as e:
        eng.chain_count()
    assert e.value.code == MS_ERR_ARG and "position 10 of contig 0" in e.value.message
    with pytest.raises(MutSimError) as e:
        eng.chain_write([1, 2])
    assert e.value.code == MS_ERR_ARG
    recs[0]["src"] = 50
    eng.load_records(recs)
    eng.apply()
    assert list(eng.chain_count()) == [2, 1]
    from mutation_simulator_b200._lib import MS_ERR_LIMIT
    with pytest.raises(MutSimError) as e:
        eng.chain_write([2 ** 31 - 2, 2 ** 31])
    assert e.value.code == MS_ERR_LIMIT
    eng.adopt_output()
    with pytest.raises(MutSimError) as e:
        eng.chain_count()
    assert e.value.code == MS_ERR_STATE
    eng.close()


def test_replay_of_a_runs_vcf_gives_its_chain_without_the_tli_copies():
    """A sampled run's chain, and the chain of replaying its VCF body: TLI inserts come back as literals (the VCF
    does not record their source), so their copy chains go and the ids close up; unpaired translocation halves (no-op
    records) are not in the VCF and change nothing."""
    rng = np.random.default_rng(4)
    lens = (70_001, 16_384, 40_000, 33_000, 16_383)
    genome = [(b"c%d" % i, b"c%d x" % i, rng.choice(np.frombuffer(b"ACGT", np.uint8), n).tobytes(), 60) for i, n in enumerate(lens)]
    eng, _, _, L = engine_for(genome)
    rates = [0.01, 0.002, 0.002, 0.001, 0.001, 0.001, 0.001]
    cdf = (np.cumsum(rates) / sum(rates)).tolist()
    cdf[-1] = 1.0
    ranges = [dict(contig=i, start=0, stop=int(n) - 1, k=int(int(n) * sum(rates)), limit=int(n), cdf=cdf,
                   minlen=[1, 1, 1, 24, 1, 1, 1], maxlen=[1, 10, 10, 50, 50, 50, 50]) for i, n in enumerate(L)]
    eng.set_ranges(ranges, [1] * 7, 1, 2.0 / 3.0)         # inversions of >= 24 bases: none equals its reverse complement
    eng.sample(21)
    eng.apply()
    recs = eng.records(True)
    assert (recs["type"] == R.T_TLI).any() and (recs["type"] == R.T_IV).any()
    text, _, _ = device_chain(eng)
    body = eng.vcf()
    # the run's chains, contig by contig: primary, then copies in record order; drop the TLI copies
    kept = []
    for c in range(len(lens)):
        own = [ch for ch in parse_chains(text) if ch["qname"] == "c%d" % c]
        copies = recs[(recs["contig"] == c) & np.isin(recs["kind"], (R.K_RAW, R.K_CONV, R.K_RC)) & (recs["prod"] > 0)]
        prim = own[:len(own) - len(copies)]
        kept += prim + [ch for ch, r in zip(own[len(prim):], copies) if r["type"] != R.T_TLI]
    assert eng.load_vcf(body)
    eng.apply()
    replay = parse_chains(device_chain(eng)[0])
    assert len(replay) == len(kept)
    for a, b in zip(replay, kept):
        assert {k: v for k, v in a.items() if k != "id"} == {k: v for k, v in b.items() if k != "id"}
    assert [c["id"] for c in replay] == list(range(1, len(replay) + 1))
    eng.close()


# ---- command line ----------------------------------------------------------------------------------------------------
SV_ARGS = ["args", "-sn", "0.01", "-in", "0.004", "-inmax", "9", "-de", "0.004", "-demax", "20", "-iv", "0.003", "-ivmax", "30",
           "-du", "0.003", "-dumax", "20", "-tl", "0.003", "-tlmax", "20"]


def _read(p):
    b = p.read_bytes()
    return gzip.decompress(b) if p.suffix == ".gz" else b


def _vcf_snps(vcf: bytes):
    out = {}
    for ln in vcf.decode().splitlines():
        f = ln.split("\t")
        if ln.startswith("#") or f[7] != ".":
            continue
        out.setdefault(f[0], []).append(int(f[1]) - 1)
    return out


def _lift_cli(tmp_path, prefix):
    ins = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / "in.fa")}
    outs = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / f"{prefix}_ms.fa")}
    chains = parse_chains((tmp_path / f"{prefix}_ms.chain").read_bytes())
    lift_check(chains, ins, outs, _vcf_snps((tmp_path / f"{prefix}_ms.vcf").read_bytes()), partition=False)
    return chains


@pytest.mark.parametrize("mode", ["args", "rmt"])
def test_cli_chain_lifts_the_devices_own_output(tmp_path, mode):
    if mode == "args":
        shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
        tail = SV_ARGS
    else:
        shutil.copy(GOLDEN / "rmt_ranges" / "in.fa", tmp_path / "in.fa")
        shutil.copy(GOLDEN / "rmt_ranges" / "in.rmt", tmp_path / "in.rmt")
        tail = ["rmt", tmp_path / "in.rmt"]
    run_main([tmp_path / "in.fa", "-o", tmp_path / "a", "-q", "-w", "--seed", "3", "--chain"] + tail)
    chains = _lift_cli(tmp_path, "a")
    assert any(c["qstrand"] == "-" for c in chains) or mode == "rmt"
    run_main([tmp_path / "in.fa", "-o", tmp_path / "b", "-q", "-w", "--seed", "3"] + tail)
    assert not (tmp_path / "b_ms.chain").exists()                 # no --chain: no chain file, same outputs
    assert (tmp_path / "b_ms.fa").read_bytes() == (tmp_path / "a_ms.fa").read_bytes()


@pytest.mark.parametrize("bgzip", [False, True])
def test_cli_modes_write_their_chains(tmp_path, bgzip):
    z, gz = (["--bgzip"], ".gz") if bgzip else ([], "")
    shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
    run_main([tmp_path / "in.fa", "-o", tmp_path / "a", "-q", "-w", "--seed", "5", "--chain"] + z + SV_ARGS)
    run_main([tmp_path / "in.fa", "-o", tmp_path / "p", "-q", "-w", "--seed", "5", "--chain"] + SV_ARGS)
    plain = (tmp_path / "p_ms.chain").read_bytes()
    assert len(plain) > 0 and _read(tmp_path / f"a_ms.chain{gz}") == plain
    # vcf replay: the run's chain without its TLI copy chains (checked on the engine above); here: it is written
    run_main([tmp_path / "in.fa", "-o", tmp_path / "v", "-q", "--chain"] + z + ["vcf", tmp_path / f"a_ms.vcf{gz}"])
    assert parse_chains(_read(tmp_path / f"v_ms.chain{gz}"))
    # it
    shutil.copy(GOLDEN / "it_basic" / "in.fa", tmp_path / "it.fa")
    run_main([tmp_path / "it.fa", "-o", tmp_path / "i", "-q", "-w", "--seed", "5", "--chain"] + z + ["it", "0.004"])
    assert not (tmp_path / f"i_ms.chain{gz}").exists()
    it_text = _read(tmp_path / f"i_ms_it.chain{gz}")
    src = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / "it.fa")}
    out = {c[0].decode(): c[2] for c in read_fasta_simple(tmp_path / "i_ms_it.fa")} if not bgzip else None
    if out is not None:
        lift_check(parse_chains(it_text), src, out)
    # rmt with IT, chained in HBM and through the reloaded *_ms.fa
    shutil.copy(GOLDEN / "rmt_it" / "in.fa", tmp_path / "r.fa")
    shutil.copy(GOLDEN / "rmt_it" / "in.rmt", tmp_path / "r.rmt")
    run_main([tmp_path / "r.fa", "-o", tmp_path / "h", "-q", "-w", "--seed", "9", "--chain"] + z + ["rmt", tmp_path / "r.rmt"])
    run_main([tmp_path / "r.fa", "-o", tmp_path / "n", "-q", "-w", "--seed", "9", "--chain"] + z + ["rmt", tmp_path / "r.rmt"],
             env={"MS_NO_CHAIN": "1"})
    for f in (f"_ms.chain{gz}", f"_ms_it.chain{gz}"):
        assert (tmp_path / ("h" + f)).read_bytes() == (tmp_path / ("n" + f)).read_bytes(), f
        assert parse_chains(_read(tmp_path / ("h" + f)))


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_multi_gpu_chain_equals_single_gpu(tmp_path):
    from tests.test_gpu_multi import make_genome
    n = min(_ngpu(), 4)
    make_genome(tmp_path / "g.fa", [90_000, 70_011, 65_000, 40_000, 33_333, 20_000, 7, 1_000], 1)
    argv = ["-q", "--seed", "5", "--chain", "args", "-sn", "0.01", "-in", "0.002", "-de", "0.002", "-du", "0.002", "-iv",
            "0.002", "-tl", "0.002"]
    for d, k, env, port in (("a", 1, {}, 0), ("b", n, {}, 29653), ("c", n, {"MS_SHARD": "tiles"}, 29654)):
        (tmp_path / d).mkdir()
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "g")] + argv, k, port, **env)
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "z"), "--bgzip"] + argv, k, port + 10 if port else 0, **env)
    want = (tmp_path / "a" / "g_ms.chain").read_bytes()
    assert len(want) > 0
    for d in ("b", "c"):
        assert (tmp_path / d / "g_ms.chain").read_bytes() == want, d
        assert gzip.decompress((tmp_path / d / "z_ms.chain.gz").read_bytes()) == want, d
