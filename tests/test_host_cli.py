"""The C++ host (`main compress|decompress <src> <dst>`) against the reference: the archives its unmodified binary wrote for
the edge-case tree (tests/golden/), and its reader restated (oracle_lib.ref_decompress, pinned to what the binary wrote when
it read those archives, tests/test_oracle.py).

`[emu]`: the host sources linked against the SIMT-emulator build of the C ABI (CPU, here). `[cuda]`: the shipped `main`
over libzwz_cuda.so on the B200. Criteria from BASELINE.json:
  (1) the reference decompresses OUR archives to the original bytes, "MD5 match" on every file;
  (2) WE decompress the REFERENCE's archives to bytes identical to the reference's own decompression (including the short
      output of its truncated records) and print the same verdicts;
  (3) the MD5 stored in our records is the reference's (OpenSSL) digest of the source file;
  and the `.zwz` layout / archive naming / size-descending round-robin deal are the reference's.
"""
import filecmp
import hashlib
import json
import os
import shutil
import subprocess

import pytest

import oracle_lib as O
import zwz_format
from tools import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
HOST = os.path.join(ROOT, "parallel-data-compression-and-decompression_b200", "host")


@pytest.fixture(params=[pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)])
def main_bin(request):
    if request.param == "emu":
        subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "simt"), "hostemu/main"], check=True, capture_output=True,
                       env={k: v for k, v in os.environ.items() if k not in ("CC", "CXX")})
        return os.path.join(ROOT, "tests", "simt", "hostemu", "main")
    p = os.path.join(HOST, "main")
    assert os.path.exists(p), "build the host first (__graft_entry__.build())"
    return p


def run(cmd, env=None, check=True):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run(cmd, env=e, capture_output=True, text=True)
    if check:
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout + r.stderr


def same_tree(a, b):
    c = filecmp.dircmp(a, b)
    stack = [c]
    while stack:
        d = stack.pop()
        assert not d.left_only and not d.right_only, (d.left_only, d.right_only)
        for f in d.common_files:
            assert filecmp.cmp(os.path.join(d.left, f), os.path.join(d.right, f), shallow=False), f
        stack += list(d.subdirs.values())


@pytest.fixture
def edge_tree(tmp_path):
    src = tmp_path / "work" / "edge"
    src.mkdir(parents=True)
    specs = corpus.edge_case_tree(str(src))
    return str(src), specs


def reference_archives_of(src, name):
    """The archives the reference binary wrote for the edge-case tree (edge_r1: one rank, edge_r2: two), once it is checked
    that `src` is that very tree."""
    man = json.load(open(os.path.join(GOLD, "manifest.json")))
    assert O.md5_tree(src) == man["inputs"]
    return os.path.join(GOLD, name)


def test_reference_decompresses_our_archive(main_bin, edge_tree, tmp_path):
    src, specs = edge_tree
    arch = str(tmp_path / "arch")
    log = run([main_bin, "compress", src, arch])
    assert "Operation: compress" in log and "Processor Count: 1" in log and "Time Taken:" in log
    assert os.listdir(arch) == ["compressed_0.zwz"]                       # compression.cpp:151-159
    assert os.path.exists(os.path.join(os.path.dirname(src), "sorted_files_by_size.txt"))  # file_sort.cpp:33
    out = str(tmp_path / "out")
    assert O.ref_decompress(arch, out) == {"match": len(specs), "mismatch": 0}
    same_tree(src, out)  # lossless even for the incompressible 65 535-byte chunk the reference itself truncates


def test_record_layout_and_md5(main_bin, edge_tree, tmp_path):
    src, specs = edge_tree
    arch = str(tmp_path / "arch")
    run([main_bin, "compress", src, arch])
    recs = zwz_format.parse(open(os.path.join(arch, "compressed_0.zwz"), "rb").read())
    order = open(os.path.join(os.path.dirname(src), "sorted_files_by_size.txt")).read().split("\n")[:-1]
    sizes = {s.relpath: s.size for s in specs}
    assert [sizes[p] for p in order] == sorted(sizes.values(), reverse=True)          # size-descending
    seen = []
    by = {}
    for r in recs:
        if not seen or seen[-1] != r.path:
            seen.append(r.path)
        by.setdefault(r.path, []).append(r)
    assert seen == order                                                              # records in file order, contiguous
    for p, rs in by.items():
        assert [r.seq for r in rs] == list(range(len(rs)))                            # 0..n-1
        assert [r.last for r in rs] == [False] * (len(rs) - 1) + [True]
        assert all(len(r.payload) <= 65535 for r in rs)                               # decompression.cpp:116
        assert rs[-1].md5.decode() == hashlib.md5(open(os.path.join(src, p), "rb").read()).hexdigest()
        assert len(rs) >= sizes[p] // 65535 + 1                                        # chunking rule (+1 per split chunk)
    assert len(by["rand70k.bin"]) == 3                 # 65 535 incompressible -> split in two, + the 4 465-byte tail
    assert len(by["exact65535.txt"]) == 2 and len(by["exact65535.txt"][1].payload) == 8   # empty tail chunk 78 9c 03 00 00 00 00 01
    assert len(by["empty.bin"]) == 1


def test_we_decompress_reference_archives_byte_exact(main_bin, edge_tree, tmp_path):
    src, specs = edge_tree
    arch = reference_archives_of(src, "edge_r1")
    ref_out, our_out = str(tmp_path / "ref_out"), str(tmp_path / "our_out")
    rv = O.ref_decompress(arch, ref_out)
    olog = run([main_bin, "decompress", arch, our_out])
    same_tree(ref_out, our_out)
    assert (olog.count("MD5 match for file"), olog.count("MD5 mismatch for file")) == (rv["match"], rv["mismatch"])
    assert olog.count("MD5 mismatch for file") == 1   # the reference's own truncated record (SURVEY.md §5.1)


@pytest.mark.parametrize("name", ["edge_r1", "edge_r2", "foreign"])
def test_we_decompress_golden_archives(main_bin, name, tmp_path):
    """Same check against the committed archives (no reference binary needed at run time)."""
    man = json.load(open(os.path.join(GOLD, "manifest.json")))
    out = str(tmp_path / "out")
    log = run([main_bin, "decompress", os.path.join(GOLD, name), out])
    got = {}
    for d, _, files in os.walk(out):
        for f in files:
            p = os.path.join(d, f)
            b = open(p, "rb").read()
            got[os.path.relpath(p, out)] = {"size": len(b), "md5": hashlib.md5(b).hexdigest()}
    assert got == man[name]["outputs"]
    assert log.count("MD5 match for file") == man[name]["verdicts"]["match"]
    assert log.count("MD5 mismatch for file") == man[name]["verdicts"]["mismatch"]


def test_self_launch_one_process_per_gpu(main_bin, edge_tree, tmp_path):
    """`ZWZ_GPUS=2 main compress` forks rank 1 itself (no MPI launcher): two archives with the reference's deal, and the
    reference's reader reads them back to the source tree."""
    src, specs = edge_tree
    arch, out = str(tmp_path / "arch"), str(tmp_path / "out")
    log = run([main_bin, "compress", src, arch], {"ZWZ_GPUS": "2"})
    assert sorted(f for f in os.listdir(arch) if f.endswith(".zwz")) == ["compressed_0.zwz", "compressed_1.zwz"]
    assert "Processor Count: 2" in log and not os.path.exists(os.path.join(arch, ".zwz_record_ready"))
    order = sorted(specs, key=lambda s: -s.size)
    for r in (0, 1):
        paths = []
        for rec in zwz_format.parse(open(os.path.join(arch, f"compressed_{r}.zwz"), "rb").read()):
            if rec.path not in paths:
                paths.append(rec.path)
        assert sorted(paths) == sorted(s.relpath for s in order[r::2])
    O.ref_decompress(arch, out)
    same_tree(src, out)


def test_strict_mode_names_the_records_zlib_would_have_rejected(main_bin, tmp_path):
    """ZWZ_STRICT=1 (SURVEY.md §8(f) rank 3): the reference ignores zlib's return codes (decompression.cpp:31); with the flag
    every record that does not reach a clean end of stream is named and the exit code is 4. Same bytes are written either way.
    The golden 1-rank archive holds the reference's own truncated records (incompressible 65 535-byte chunks, §5.1)."""
    import oracle_lib as O
    recs = zwz_format.parse(open(os.path.join(GOLD, "edge_r1", "compressed_0.zwz"), "rb").read())
    bad = [(r.path, r.seq) for r in recs if O.inflate(r.payload, 70000)[1] != O.STREAM_END]
    assert bad, "fixture lost its truncated records"
    out1, out2 = str(tmp_path / "o1"), str(tmp_path / "o2")
    r = subprocess.run([main_bin, "decompress", os.path.join(GOLD, "edge_r1"), out1], env={**os.environ, "ZWZ_STRICT": "1"}, capture_output=True, text=True)
    assert r.returncode == 4, r.stderr[-2000:]
    named = [l for l in r.stderr.splitlines() if l.startswith("Corrupt record: ")]
    assert sorted(named) == sorted(f"Corrupt record: {p} sequence {q} (truncated stream)" for p, q in bad)
    log = run([main_bin, "decompress", os.path.join(GOLD, "edge_r1"), out2])      # default: the reference's silence, exit 0
    assert "Corrupt record" not in log
    same_tree(out1, out2)


def test_two_ranks_same_deal_as_reference(main_bin, edge_tree, tmp_path):
    """`mpirun -n 2` analogue: rank r takes sorted files r, r+2, ... and writes compressed_<r>.zwz (compression.cpp:31-41,157)."""
    src, specs = edge_tree
    ours, ref = str(tmp_path / "ours"), reference_archives_of(src, "edge_r2")
    procs = [subprocess.Popen([main_bin, "compress", src, ours], env={**os.environ, "ZWZ_WORLD": "2", "ZWZ_RANK": str(r)},
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in (0, 1)]
    for p in procs:
        p.communicate()
        assert p.returncode == 0
    assert sorted(os.listdir(ours)) == sorted(os.listdir(ref)) == ["compressed_0.zwz", "compressed_1.zwz"]
    for a in ("compressed_0.zwz", "compressed_1.zwz"):
        po = [r.path for r in zwz_format.parse(open(os.path.join(ours, a), "rb").read()) if r.seq == 0]
        pr = [r.path for r in zwz_format.parse(open(os.path.join(ref, a), "rb").read()) if r.seq == 0]
        assert po == pr, a
    out = str(tmp_path / "out")
    assert O.ref_decompress(ours, out)["match"] == len(specs)
    same_tree(src, out)


def test_self_round_trip_and_multi_batch(main_bin, tmp_path):
    """Small batches force many GPU round trips and the large-file streaming path (segments + chained MD5)."""
    src = tmp_path / "w" / "src"
    src.mkdir(parents=True)
    specs = corpus.c1_specs(12, seed=599, min_size=2000, max_size=300_000)
    specs.append(corpus.FileSpec("big/huge.log", 4_400_000, "T", 999))   # > 64 chunks => segmented path with ZWZ_BATCH_MB=1
    corpus.write_tree(str(src), specs, 599)
    arch, out = str(tmp_path / "arch"), str(tmp_path / "out")
    run([main_bin, "compress", str(src) + "/", arch + "/"], {"ZWZ_BATCH_MB": "1"})   # trailing slashes are stripped (main.cpp:72-76)
    log = run([main_bin, "decompress", arch, out], {"ZWZ_BATCH_MB": "1"})
    assert log.count("MD5 match for file") == len(specs) and "mismatch" not in log
    same_tree(str(src), out)
    # the worker pool (host/pipeline.hpp) commits batches in order: same archive bytes and same console lines for any W
    arch1, out1 = str(tmp_path / "arch1"), str(tmp_path / "out1")
    run([main_bin, "compress", str(src), arch1], {"ZWZ_BATCH_MB": "1", "ZWZ_WORKERS": "1"})
    assert filecmp.cmp(os.path.join(arch, "compressed_0.zwz"), os.path.join(arch1, "compressed_0.zwz"), shallow=False)
    log1 = run([main_bin, "decompress", arch1, out1], {"ZWZ_BATCH_MB": "1", "ZWZ_WORKERS": "1"})
    verdicts = lambda t, o: [l.replace(o, "") for l in t.splitlines() if l.startswith("MD5 match")]  # noqa: E731
    assert verdicts(log, out) == verdicts(log1, out1)
    same_tree(str(src), out1)


def _small_tree(tmp_path, with_big=True):
    src = tmp_path / "w" / "src"
    src.mkdir(parents=True)
    specs = corpus.c1_specs(10, seed=601, min_size=2000, max_size=200_000)
    if with_big:
        specs.append(corpus.FileSpec("big/huge.log", 3_300_000, "T", 998))   # cut into segments with ZWZ_BATCH_MB=1
    corpus.write_tree(str(src), specs, 601)
    return str(src), specs


def test_stale_marker_of_a_killed_run_is_not_trusted(main_bin, tmp_path):
    """ADVICE r1: a `.zwz_record_ready` left by a killed run (plus its old record file) must not let rank 1 deal from the old
    list when it starts before rank 0. The marker carries the run id; a rank without its run's marker fails after the
    rendezvous timeout instead of exiting 0."""
    src, specs = _small_tree(tmp_path, with_big=False)
    arch = tmp_path / "arch"
    arch.mkdir()
    record = os.path.join(os.path.dirname(src), "sorted_files_by_size.txt")
    open(record, "w").write("\n".join(s.relpath for s in specs[:3]) + "\n")          # what the killed run left: a partial list
    (arch / ".zwz_record_ready").write_text("killed-run\n" + record + "\n")
    env = {**os.environ, "ZWZ_WORLD": "2", "ZWZ_RUN_ID": "run-42", "ZWZ_RENDEZVOUS_TIMEOUT": "60"}
    p1 = subprocess.Popen([main_bin, "compress", src, str(arch)], env={**env, "ZWZ_RANK": "1"}, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    import time
    time.sleep(1.0)                                                                      # rank 1 is polling; the stale marker is all there is
    assert p1.poll() is None
    p0 = subprocess.Popen([main_bin, "compress", src, str(arch)], env={**env, "ZWZ_RANK": "0"}, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    for p in (p0, p1):
        p.communicate()
        assert p.returncode == 0
    got = set()
    for a in ("compressed_0.zwz", "compressed_1.zwz"):
        got |= {r.path for r in zwz_format.parse(open(os.path.join(str(arch), a), "rb").read())}
    assert got == {s.relpath for s in specs}                                             # nothing dealt from the stale list
    # and alone, with only a foreign marker to look at, a rank gives up with a non-zero exit code
    r = subprocess.run([main_bin, "compress", src, str(arch)], env={**env, "ZWZ_RANK": "1", "ZWZ_RUN_ID": "run-43", "ZWZ_RENDEZVOUS_TIMEOUT": "1"},
                       capture_output=True, text=True)
    assert r.returncode != 0 and "timed out" in r.stderr


def test_generic_rank_variables_do_not_shard(main_bin, tmp_path):
    """ADVICE r1: RANK/WORLD_SIZE of an enclosing torch/k8s job must not turn a plain run into rank r of N."""
    src, specs = _small_tree(tmp_path, with_big=False)
    arch = str(tmp_path / "arch")
    log = run([main_bin, "compress", src, arch], {"RANK": "1", "WORLD_SIZE": "4", "LOCAL_RANK": "1"})
    assert "Processor Count: 1" in log and os.listdir(arch) == ["compressed_0.zwz"]
    assert {r.path for r in zwz_format.parse(open(os.path.join(arch, "compressed_0.zwz"), "rb").read())} == {s.relpath for s in specs}


def test_verify_all_gives_the_verdict_the_reference_skips(main_bin, tmp_path):
    """decompression.cpp:132 only judges a file when its is_last record arrives in order; the hand-built foreign archive has a
    file whose last record comes first. ZWZ_VERIFY_ALL=1 prints a verdict for every complete file."""
    man = json.load(open(os.path.join(GOLD, "manifest.json")))
    o1, o2 = str(tmp_path / "o1"), str(tmp_path / "o2")
    base = run([main_bin, "decompress", os.path.join(GOLD, "foreign"), o1])
    full = run([main_bin, "decompress", os.path.join(GOLD, "foreign"), o2], {"ZWZ_VERIFY_ALL": "1"})
    n_files = len(man["foreign"]["outputs"])
    assert base.count("MD5 match for file") + base.count("MD5 mismatch for file") == man["foreign"]["verdicts"]["match"] + man["foreign"]["verdicts"]["mismatch"] < n_files
    assert full.count("MD5 match for file") + full.count("MD5 mismatch for file") == n_files
    same_tree(o1, o2)


def test_quarantine_moves_mismatching_files_to_bad(main_bin, tmp_path):
    """README.md:175,186 promise a bad/ directory for files whose MD5 does not match; the reference's code leaves them in place
    (and so does the default). ZWZ_QUARANTINE=1 moves them. The golden 1-rank archive holds the reference's own lossy record."""
    man = json.load(open(os.path.join(GOLD, "manifest.json")))
    assert man["edge_r1"]["verdicts"]["mismatch"] == 1
    out = str(tmp_path / "out")
    log = run([main_bin, "decompress", os.path.join(GOLD, "edge_r1"), out], {"ZWZ_QUARANTINE": "1"})
    assert log.count("MD5 mismatch for file") == 1 and "Moved to: " in log
    bad = [os.path.relpath(os.path.join(d, f), os.path.join(out, "bad")) for d, _, fs_ in os.walk(os.path.join(out, "bad")) for f in fs_]
    assert bad == ["rand70k.bin"] and not os.path.exists(os.path.join(out, "rand70k.bin"))
    b = open(os.path.join(out, "bad", "rand70k.bin"), "rb").read()
    assert {"size": len(b), "md5": hashlib.md5(b).hexdigest()} == man["edge_r1"]["outputs"]["rand70k.bin"]


@pytest.mark.parametrize("launch", ["ranks", "self"])
def test_multi_rank_decompress(main_bin, tmp_path, launch):
    """SURVEY.md §8(f)4: the reference decompresses on rank 0 only (main.cpp:61-69). Here the batches — whole small files and
    record ranges of a large one (segments, offsets through the shared ledger) — are dealt over the ranks: two ranks started by
    a launcher (ZWZ_RANK/ZWZ_WORLD) or forked by `ZWZ_GPUS=2 main decompress`; same tree, one verdict per file."""
    src, specs = _small_tree(tmp_path)
    arch, out = str(tmp_path / "arch"), str(tmp_path / "out")
    run([main_bin, "compress", src, arch], {"ZWZ_GPUS": "2", "ZWZ_BATCH_MB": "1"})
    if launch == "self":
        log = run([main_bin, "decompress", arch, out], {"ZWZ_GPUS": "2", "ZWZ_BATCH_MB": "1"})
        assert "Processor Count: 2" in log
    else:
        env = {**os.environ, "ZWZ_WORLD": "2", "ZWZ_BATCH_MB": "1", "ZWZ_RUN_ID": "d1"}
        procs = [subprocess.Popen([main_bin, "decompress", arch, out], env={**env, "ZWZ_RANK": str(r)}, stdout=subprocess.PIPE,
                                  stderr=subprocess.STDOUT, text=True) for r in (0, 1)]
        log = ""
        for p in procs:
            log += p.communicate()[0]
            assert p.returncode == 0
    assert log.count("MD5 match for file") == len(specs) and "mismatch" not in log
    assert not os.path.exists(os.path.join(out, ".zwz_segments")) or launch == "ranks"
    shutil.rmtree(os.path.join(out, ".zwz_segments"), ignore_errors=True)
    same_tree(src, out)


@pytest.mark.parametrize("launch", ["self", "ranks"])
def test_one_file_cut_over_the_ranks_lands_in_one_archive(main_bin, tmp_path, launch):
    """BASELINE config 3 / SURVEY.md §8(e): the reference's deal is file-granular (compression.cpp:31-41) and its reader wants
    all records of a path in ONE archive (decompression.cpp:52-55). A file that is cut into segments is deflated by several
    ranks here; the owner hands out archive offsets and sequence ids through the segment ledger and every rank writes its
    records into the owner's archive. The reference's reader reads the result back."""
    src = tmp_path / "w" / "src"
    src.mkdir(parents=True)
    specs = [corpus.FileSpec("big/huge.log", 5_300_000, "T", 997), corpus.FileSpec("big/second.bin", 2_500_000, "S", 996),
             corpus.FileSpec("small/a.txt", 70_000, "T", 995), corpus.FileSpec("small/r.bin", 140_000, "R", 994)]
    corpus.write_tree(str(src), specs, 603)
    arch, out = str(tmp_path / "arch"), str(tmp_path / "out")
    if launch == "self":
        run([main_bin, "compress", str(src), arch], {"ZWZ_GPUS": "3", "ZWZ_BATCH_MB": "1"})
    else:
        env = {**os.environ, "ZWZ_WORLD": "3", "ZWZ_BATCH_MB": "1", "ZWZ_RUN_ID": "c3"}
        procs = [subprocess.Popen([main_bin, "compress", str(src), arch], env={**env, "ZWZ_RANK": str(r)}, stdout=subprocess.PIPE,
                                  stderr=subprocess.STDOUT, text=True) for r in (2, 1, 0)]
        for p in procs:
            o = p.communicate()[0]
            assert p.returncode == 0, o[-2000:]
    assert sorted(f for f in os.listdir(arch)) == ["compressed_0.zwz", "compressed_1.zwz", "compressed_2.zwz"]   # ledger and marker are gone
    owner = {}
    for r in range(3):
        recs = zwz_format.parse(open(os.path.join(arch, f"compressed_{r}.zwz"), "rb").read())
        by = {}
        for rec in recs:
            by.setdefault(rec.path, []).append(rec)
        for pth, rs in by.items():
            assert pth not in owner                                          # all records of a path in one archive
            owner[pth] = r
            assert [x.seq for x in rs] == list(range(len(rs)))               # contiguous ids, in order
            assert [x.last for x in rs] == [False] * (len(rs) - 1) + [True]
            assert rs[-1].md5.decode() == hashlib.md5(open(os.path.join(str(src), pth), "rb").read()).hexdigest()
    order = sorted(specs, key=lambda s_: -s_.size)
    assert owner == {s_.relpath: i % 3 for i, s_ in enumerate(order)}       # the reference's deal decides the archive
    assert O.ref_decompress(arch, out) == {"match": len(specs), "mismatch": 0}
    same_tree(str(src), out)


def test_usage_and_errors(main_bin, tmp_path):
    r = subprocess.run([main_bin, "compress"], capture_output=True, text=True)
    assert r.returncode != 0 and "Usage:" in r.stderr
    r = subprocess.run([main_bin, "compress", str(tmp_path / "nope"), str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "Source path does not exist." in r.stderr
    (tmp_path / "s").mkdir()
    r = subprocess.run([main_bin, "frobnicate", str(tmp_path / "s"), str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "Invalid operation" in r.stderr
