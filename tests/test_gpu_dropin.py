"""GPU: the reference's own construct.cc (compiled in place, tests/cpp/Makefile)
running on the B200 engine through the ram::MinimizerEngine facade, and our
batched FindOverlapsAndCreatePiles replacement with the reference signature -
both against the CPU oracle, bit exact."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from raven_b200 import synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
BIN = os.path.join(HERE, "cpp", "_build", "dropin_test")
REF_META = json.load(open(os.path.join(HERE, "golden", "reference_golden.json")))
REF_GOLD = np.load(os.path.join(HERE, "golden", "reference_golden.npz"))


def reference_assembly():
    """RavenTest.Assemble's polished unitigs from the reference's own sources over the
    CPU oracle (stored by tests/golden/make_reference_golden.py): names and sequences."""
    names = REF_META["assemble_rounds2_names"]
    return names, [REF_GOLD[f"assemble_rounds2_unitig{i}"].tobytes() for i in range(len(names))]


def write_vec(f, a):
    f.write(struct.pack("<Q", a.size))
    f.write(np.ascontiguousarray(a).tobytes())


def read_vec(f, dt):
    (n,) = struct.unpack("<Q", f.read(8))
    return np.frombuffer(f.read(n * np.dtype(dt).itemsize), dtype=dt).copy()


def run_dropin(tmp_path, rs, k, w, freq, kmax, minhash):
    if not os.path.exists(BIN):
        pytest.skip("tests/cpp/_build/dropin_test not built (needs the reference's sources at build time)")
    inp, out = str(tmp_path / "reads.bin"), str(tmp_path / "out.bin")
    with open(inp, "wb") as f:
        write_vec(f, rs.words.astype(np.uint64))
        write_vec(f, rs.word_off.astype(np.uint64))
        write_vec(f, rs.lens.astype(np.uint32))
    subprocess.run([BIN, inp, out, str(k), str(w), str(freq), str(kmax), str(int(minhash))],
                   check=True, stderr=subprocess.DEVNULL, timeout=600)
    res = []
    with open(out, "rb") as f:
        for _ in range(2):
            res.append(dict(overlaps=read_vec(f, np.uint32).reshape(-1, 8),
                            ovl_off=read_vec(f, np.uint64), pile=read_vec(f, np.uint16),
                            pile_off=read_vec(f, np.uint64)))
    return res


@pytest.mark.parametrize("minhash", [False, True])
def test_reference_construct_on_b200_facade(tmp_path, oracle, lambda_reads, minhash):
    a, b = run_dropin(tmp_path, lambda_reads, 15, 5, 0.001, 32, minhash)
    want = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(lambda_reads),
                         0.001, 32, minhash)
    for got, name in ((a, "reference construct.cc over the facade"),
                      (b, "batched replacement")):
        for key in ("overlaps", "ovl_off", "pile", "pile_off"):
            assert np.array_equal(got[key], want[key]), (name, key)


def test_dropin_synthetic_small_kmax(tmp_path, oracle):
    rs = synth.make_reads(40_000, 150, 3000, seed=13)
    a, b = run_dropin(tmp_path, rs, 15, 5, 0.001, 6, False)
    want = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), 0.001, 6, False)
    for got in (a, b):
        for key in ("overlaps", "ovl_off", "pile", "pile_off"):
            assert np.array_equal(got[key], want[key]), key


def test_full_pipeline_on_b200_equals_oracle_pipeline(tmp_path, oracle, lambda_reads):
    """RavenTest.Assemble with the reference's own sources on the B200 facades
    (ram::MinimizerEngine, racon::Polisher incl. GPU POA) == the same sources over
    the CPU oracle: identical polished unitig, and the reference's golden value:
    1137 edits to NC_001416 (RavenTest/src/raven_test.cpp:66)."""
    from raven_b200 import seqio
    binary = os.path.join(HERE, "cpp", "_build", "assemble_test")
    if not os.path.exists(binary):
        pytest.skip("tests/cpp/_build/assemble_test not built")
    inp, out = str(tmp_path / "reads.bin"), str(tmp_path / "unitigs.txt")
    with open(inp, "wb") as f:
        write_vec(f, lambda_reads.words.astype(np.uint64))
        write_vec(f, lambda_reads.word_off.astype(np.uint64))
        write_vec(f, lambda_reads.lens.astype(np.uint32))
        write_vec(f, lambda_reads.block_quality.astype(np.uint8))
        write_vec(f, lambda_reads.bq_off.astype(np.uint64))
    subprocess.run([binary, inp, out, "1", "2"], check=True, stderr=subprocess.DEVNULL,
                   timeout=900)
    lines = open(out).read().split("\n")
    names, seqs = lines[0:-1:2], [s.encode() for s in lines[1::2]]
    want_names, want_seqs = reference_assembly()
    assert names == want_names
    assert seqs == want_seqs
    genome = seqio.ReadSet.load(os.path.join(HERE, "golden", "lambda_genome.npz")).ascii(0)
    rc = seqs[0].translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]
    assert oracle.edit_distance(rc, genome) == 1137   # EXPECT_EQ(1137, ...) raven_test.cpp:66


@pytest.mark.parametrize("identity", [0.0, 0.8, 0.9])
def test_stage2_and_identity_filter_batched_equals_reference(tmp_path, lambda_reads, identity):
    """raven::ResolveContainedReads + raven::FindOverlapsAndRepetetiveRegions
    (construct.cc:154-246, 316-491): the reference's own functions over the facade
    (per-read Map, host edlibAlign per overlap) vs the batched B200 replacements
    (one device map per batch, rvn_edit_distance_batch): identical overlap lists
    and identical piles, field by field."""
    binary = os.path.join(HERE, "cpp", "_build", "stage2_test")
    if not os.path.exists(binary):
        pytest.skip("tests/cpp/_build/stage2_test not built")
    inp, out = str(tmp_path / "reads.bin"), str(tmp_path / "out.bin")
    with open(inp, "wb") as f:
        write_vec(f, lambda_reads.words.astype(np.uint64))
        write_vec(f, lambda_reads.word_off.astype(np.uint64))
        write_vec(f, lambda_reads.lens.astype(np.uint32))
    subprocess.run([binary, inp, out, "15", "5", "0.001", str(identity)], check=True,
                   stderr=subprocess.DEVNULL, timeout=900)
    with open(out, "rb") as f:
        a = [read_vec(f, np.uint32), read_vec(f, np.uint64), read_vec(f, np.uint32),
             read_vec(f, np.uint32)]
        b = [read_vec(f, np.uint32), read_vec(f, np.uint64), read_vec(f, np.uint32),
             read_vec(f, np.uint32)]
    for x, y, name in zip(a, b, ("overlaps", "offsets", "piles", "sequence order")):
        assert np.array_equal(x, y), name
    if identity < 0.85:
        assert a[0].size > 0                   # something survives the stage ...
    else:
        assert a[0].size == 0                  # ... but no pair of 10 % error reads is 90 % identical


def test_reference_cli_runs_on_b200(tmp_path, oracle, lambda_reads):
    """The reference's own executable (RavenExe/src/main.cc + all of RavenLib,
    unmodified; tests/cpp/Makefile `_build/raven`) over the drop-in dependencies:
    FASTQ.gz in (bioparser), overlap + layout + 2 polishing rounds on the B200,
    FASTA out - the RavenTest.Assemble configuration (-M, raven_test.cpp:50-67)
    and its golden value; then `--resume` from the checkpoint (cereal) gives the
    same answer (RavenTest.Checkpoints, raven_test.cpp:69-95)."""
    import gzip
    from raven_b200 import seqio
    binary = os.path.join(HERE, "cpp", "_build", "raven")
    if not os.path.exists(binary):
        pytest.skip("tests/cpp/_build/raven not built")
    rs = lambda_reads
    fq = tmp_path / "lambda.fastq.gz"
    with gzip.open(fq, "wt", compresslevel=1) as f:
        for i in range(rs.n):
            seq = rs.ascii(i).decode()
            bq = rs.block_quality[int(rs.bq_off[i]):int(rs.bq_off[i + 1])]
            qual = "".join(chr(33 + int(q)) * 64 for q in bq)[:len(seq)]  # same block means
            f.write(f"@{rs.names[i]} extra words\n{seq}\n+\n{qual}\n")
    run = lambda *a: subprocess.run([binary, "-t", "4", "-M", *a, str(fq)], check=True,
                                    cwd=tmp_path, stdout=subprocess.PIPE,
                                    stderr=subprocess.DEVNULL, timeout=900).stdout
    out = run("-p", "2", "-F", "graph.gfa").decode().split("\n")
    names, seqs = out[0:-1:2], [s.encode() for s in out[1::2]]
    want_names, want_seqs = reference_assembly()
    assert [n[1:] for n in names] == want_names
    assert seqs == want_seqs
    genome = seqio.ReadSet.load(os.path.join(HERE, "golden", "lambda_genome.npz")).ascii(0)
    rc = seqs[0].translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]
    assert oracle.edit_distance(rc, genome) == 1137
    assert os.path.getsize(tmp_path / "graph.gfa") > 0
    assert os.path.exists(tmp_path / "raven.cereal")
    again = run("--resume", "-p", "2").decode().split("\n")
    assert again == out
