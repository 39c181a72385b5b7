import gzip
import os
import shutil
import signal
import subprocess
import sys
import tempfile
import time
import warnings

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
GOLDEN_SETS = ["edge", "example_head", "example_tail", "hard"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device here")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def gunzip_to(name, dst_dir):
    src = os.path.join(GOLD, name + ".gz")
    dst = os.path.join(dst_dir, name)
    with gzip.open(src, "rb") as f, open(dst, "wb") as g:
        g.write(f.read())
    return dst


@pytest.fixture(scope="session")
def golden_dir(tmp_path_factory):
    """All golden fixtures unpacked into a temp dir + the generated default matrix file."""
    from elector_b200 import write_default_matrix
    d = str(tmp_path_factory.mktemp("golden"))
    for s in GOLDEN_SETS:
        for ext in ("ref.fa", "cor.fa", "unc.fa", "pir", "dump"):
            gunzip_to("%s.%s" % (s, ext), d)
    for extra in os.listdir(GOLD):
        if extra.endswith(".gz") and not os.path.exists(os.path.join(d, extra[:-3])):
            gunzip_to(extra[:-3], d)
    write_default_matrix(os.path.join(d, "blosum80.mat"))
    return d


@pytest.fixture(scope="session", autouse=True)
def service_ends_with_the_session():
    """The drop-in executables hand their work to elector_server (elector_b200/csrc/service.h), which outlives them by
    ELECTOR_SERVICE_IDLE seconds.  The session gives the server its own socket and a short idle time, and waits for it to
    leave, so that no process of the tests outlives them."""
    d = tempfile.mkdtemp(prefix="elsvc")          # short: a socket path has at most 107 bytes
    sock = os.path.join(d, "sock")
    mp = pytest.MonkeyPatch()
    mp.setenv("ELECTOR_SERVICE_SOCKET", sock)
    mp.setenv("ELECTOR_SERVICE_IDLE", "2")
    yield
    mp.undo()
    deadline = time.time() + 60
    while time.time() < deadline and service_pids(sock):
        time.sleep(0.2)
    left = service_pids(sock)
    for pid in left:       # the socket is the session's own: these servers were started by its tests
        try:
            os.kill(pid, signal.SIGTERM)
        except ProcessLookupError:
            pass
    if left:
        warnings.warn("elector_server %s did not leave within 60 s of the last test; terminated" % left)
    shutil.rmtree(d, ignore_errors=True)


def service_pids(sock):
    """pids of the elector_server processes listening on `sock` (their argv is [exe, sock])"""
    pids = []
    for p in os.listdir("/proc"):
        if not p.isdigit():
            continue
        try:
            argv = open("/proc/%s/cmdline" % p, "rb").read().split(b"\0")
        except OSError:
            continue
        if len(argv) >= 2 and argv[0].endswith(b"elector_server") and argv[1] == sock.encode():
            pids.append(int(p))
    return pids


@pytest.fixture(scope="session")
def emul_bin():
    """CPU build of the per-window device code (tests/emul/poa_emul.cu)."""
    src = os.path.join(ROOT, "tests", "emul", "poa_emul.cu")
    exe = os.path.join(ROOT, "tests", "emul", "poa_emul")
    csrc = os.path.join(ROOT, "elector_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
    if not os.path.exists(exe) or any(os.path.getmtime(exe) < os.path.getmtime(p) for p in deps):
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-arch=sm_100a", "-Wno-deprecated-gpu-targets", "-o", exe, src])
    return exe


@pytest.fixture(scope="session")
def split_emul_bin():
    """CPU build of the window-cutting device code with the reference splitter's driver around it (tests/emul/split_emul.cu)."""
    src = os.path.join(ROOT, "tests", "emul", "split_emul.cu")
    exe = os.path.join(ROOT, "tests", "emul", "split_emul")
    csrc = os.path.join(ROOT, "elector_b200", "csrc")
    deps = [src, os.path.join(csrc, "split_kernel.cuh"), os.path.join(csrc, "split_host.hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(exe) < os.path.getmtime(p) for p in deps):
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-arch=sm_100a", "-Wno-deprecated-gpu-targets", "-o", exe, src])
    return exe


def read_fasta_simple(path):
    recs, h, s = [], None, []
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if h is not None:
                    recs.append((h, "".join(s)))
                h, s = line[1:], []
            else:
                s.append(line)
    if h is not None:
        recs.append((h, "".join(s)))
    return recs


def parse_dump(path):
    """oracle/ref_harness.c text dump -> list of dict(s1, s2, n1, x1, y1, x2, y2, l2)"""
    out, cur = [], None
    with open(path) as f:
        for line in f:
            t = line.split()
            if t[0] == "W":
                cur = {}
                out.append(cur)
            elif t[0] == "S1":
                cur["s1"] = int(t[1])
            elif t[0] == "S2":
                cur["s2"], cur["n1"] = int(t[1]), int(t[2])
            elif t[0] in ("X1", "Y1", "X2", "Y2"):
                cur[t[0].lower()] = [int(v) for v in t[2:]]
            elif t[0] == "L":
                cur["l2"] = int(t[1])
    return out


def parse_pir(path):
    """PIR -> list of (headers[3], rows[3])"""
    lines = open(path).read().split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    assert len(lines) % 6 == 0
    return [((lines[i], lines[i + 2], lines[i + 4]), (lines[i + 1], lines[i + 3], lines[i + 5])) for i in range(0, len(lines), 6)]


def load_example_golden():
    import json
    return json.loads(gzip.open(os.path.join(GOLD, "example_full.json.gz")).read())


@pytest.fixture(scope="session")
def example_chain(tmp_path_factory, split_emul_bin):
    """The README example up to the `poa` inputs: reads unpacked from tests/golden/example_reads.tar.xz, sorted and
    duplicated like readAndSortFiles.py, cut into shard files by the serial CPU build of the cutting code
    (tests/emul/split_emul), whose shard files are those of the reference splitter: every one has the md5 the reference's
    has in the golden (test_example_full.py, test_split_emul.py).  -> dict(work, out, shards, gold)"""
    from oracle import example_prep as ep
    src = str(tmp_path_factory.mktemp("example_src"))
    work = str(tmp_path_factory.mktemp("example_work"))
    ep.unpack(src)
    ep.sort_and_duplicate(src, work)
    out = os.path.join(work, "out")
    rc, shards = ep.reference_split(work, out, exe=split_emul_bin)
    assert rc == 0
    return {"src": src, "work": work, "out": out, "shards": shards, "gold": load_example_golden()}


@pytest.fixture(scope="session")
def example_oracle_msa(example_chain, tmp_path_factory):
    """The example through the ORACLE chain (plain-C restatement of `poa` per shard, Donatello restated): the smsa files and the
    merged records [(header, R, C, U)] in msa.fa order.  tests/test_example_full.py holds both to the reference's md5s."""
    from oracle import oracle, tally_oracle as to
    oracle.build()
    ex = example_chain
    out = str(tmp_path_factory.mktemp("example_oracle"))
    cli = os.path.join(ROOT, "oracle", "poa_oracle_cli")
    mat = os.path.join(out, "blosum80.mat")
    import elector_b200
    elector_b200.write_default_matrix(mat)
    procs = [subprocess.Popen([cli, "-pir", "%s/smsa%d" % (out, i), "-corrected_reads_fasta", "%s/out3%d" % (ex["out"], i), "-reference_reads_fasta",
                               "%s/out1%d" % (ex["out"], i), "-uncorrected_reads_fasta", "%s/out2%d" % (ex["out"], i), "-pathMatrix", mat],
                              stdout=subprocess.DEVNULL) for i in ex["shards"]]
    for p in procs:
        assert p.wait() == 0
    recs = []
    for i in ex["shards"]:
        recs += to.merge_windows(parse_pir("%s/smsa%d" % (out, i)))
    return {"dir": out, "records": recs}


def md5_file(path):
    import hashlib
    return hashlib.md5(open(path, "rb").read()).hexdigest()
