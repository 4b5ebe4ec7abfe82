"""CPU: the C-ABI library loads and exports every symbol include/swb200.h declares; the
product fails loudly without a GPU; host-side logic (sharding, merge, reductions, synthetic
data) behaves as the reference's callers do.  No compute call runs without a GPU."""
import os
import re

import numpy as np
import pytest

import sparksmithwaterman_b200 as swb
from sparksmithwaterman_b200 import _ffi, distribution, multigpu, synth
from sparksmithwaterman_b200.build import build_native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build_native()
    return _ffi.load()


def test_header_symbols_all_exported(lib):
    with open(os.path.join(ROOT, "include", "swb200.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    declared = set(re.findall(r"\b(swb_[a-z0-9_]+)\s*\(", text))
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in swb200.h but not exported"
    assert declared == set(_ffi.SIGNATURES), declared ^ set(_ffi.SIGNATURES)
    assert lib.swb_abi_version() == 2


def test_product_does_not_touch_the_oracle():
    """oracle/ is test infrastructure: only tests/ (incl. tests/checks/), smoke() and bench.py's CPU legs use it."""
    for top in ("sparksmithwaterman_b200", "tools", "include", "java", "host"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for fn in files:
                if fn.endswith((".py", ".cu", ".cuh", ".h", ".java", ".c", ".cpp")):
                    with open(os.path.join(dirpath, fn)) as f:
                        src = f.read()
                    assert "import oracle" not in src and "sw_oracle" not in src and "from oracle" not in src, fn


def test_fails_loudly_without_gpu(lib):
    if lib.swb_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(swb.SwbError) as ei:
        swb.Engine(0)
    assert "no CUDA device" in str(ei.value)


def test_synth_shape_and_determinism():
    L = synth.ref_lengths(20000)
    assert 50 <= L.min() and L.max() <= 200000
    assert abs(np.median(L) - 1609) < 60 and abs(L.mean() - 2160) < 90        # README.md:39-40 of the reference
    a, b = synth.make_refs(50), synth.make_refs(50)
    assert a == b and all(set(r) <= set(b"ACGT") for r in a)
    r1 = synth.make_reads(40, 150, a)
    assert r1 == synth.make_reads(40, 150, a) and all(len(q) == 150 for q in r1)


def test_shard_refs_partition_and_balance():
    L = synth.ref_lengths(1000)
    for world in (1, 2, 4, 8):
        shards = [multigpu.shard_refs(L, r, world) for r in range(world)]
        assert sorted(sum(shards, [])) == list(range(1000))
        tot = [int(L[s].sum()) for s in shards]
        assert max(tot) - min(tot) <= 0.05 * max(tot)


def test_merge_best_hits_is_shard_invariant():
    rng = np.random.default_rng(0)
    n_refs, n_reads = 64, 33
    scores = rng.integers(0, 40, size=(n_refs, n_reads))
    cells = rng.integers(1, 100, size=(n_refs, n_reads, 2))
    L = rng.integers(50, 500, size=n_refs)

    def best_of(ids):
        out = np.zeros((n_reads, 4), np.int32)
        for q in range(n_reads):
            k = max(range(len(ids)), key=lambda x: (scores[ids[x], q], -x))      # first max wins
            out[q] = (scores[ids[k], q], k, *cells[ids[k], q])
        return out
    single = multigpu.localize(best_of(list(range(n_refs))), list(range(n_refs)))
    for world in (2, 4, 8):
        recs = []
        for r in range(world):
            ids = multigpu.shard_refs(L, r, world)
            recs.append(multigpu.localize(best_of(ids), ids))
        assert (multigpu.merge_best_hits(np.stack(recs)) == single).all()


def test_reductions_mirror_the_reference():
    a = (10, (["b-meta", "ACGT"], [(3, ["A", "A"])]))
    b = (12, (["a-meta", "ACGA"], []))
    c = (12, (["0-meta", "ACGC"], []))
    best, opt = distribution.NoDistribution.reduce([a, b, c])
    assert best == 12 and [v[0][0] for v in opt] == ["0-meta", "a-meta"]
    # the driver as written keys on the FIRST element of each file (Distribution.java:342)
    best, opt = distribution.DistributeReference.reduce([[a, b, c]])
    assert best == 10 and [v[0][0] for v in opt] == ["b-meta"]
    sites = [(5, ["x", "1"]), (2, ["y", "2"]), (5, ["z", "3"]), (2, ["w", "4"])]
    assert [s[1][1] for s in distribution.match_site_sort(sites)] == ["2", "4", "1", "3"]     # stable
    assert distribution.wrap32(2**31 - 1 + 5) == -(2**31) + 4


def test_file_formats_mirror_inoutops(tmp_path):
    from sparksmithwaterman_b200 import inout
    rp = tmp_path / "refs.fa"
    rp.write_text(">gi|1|a\nACGT \nac gt\n>gi|2|b\n>gi|3|c\nTTTT\r\nGG\n")
    refs = inout.get_ref_seqs(str(rp))
    assert refs == [[">gi|1|a", "ACGT ac gt"], [">gi|2|b", ""], [">gi|3|c", "TTTTGG"]]      # lines not trimmed
    ip = tmp_path / "reads.txt"
    ip.write_text(">gi header\n  ACGT \n\nTT\t\n")
    assert inout.get_reads(str(ip)) == ["ACGT", "", "TT"]                                    # trimmed, empty kept
    ip.write_text("ACGT\nGG")
    assert inout.get_reads(str(ip)) == ["ACGT", "GG"]                                        # first line is a read
    with pytest.raises(ValueError):
        bad = tmp_path / "bad.fa"; bad.write_text("ACGT\n>gi|1\nAC\n"); inout.get_ref_seqs(str(bad))
    txt = inout.get_output_str(["ACGT"], (2, 1), 20, 7, [([">gi|1|a", "ACGT"], [(1, ["ACGT", "ACGT"])])])
    assert txt == ("Execution Time = 7 ms\n\n# Reference Sequences = 2\n# Reads = 1\n\nInput:\nACGT\n\n"
                   "Maximum alignment score = 20\nReference:\n>gi|1|a\nACGT\n\n\tIndex = 1\n\tACGT\n\tACGT\n\n")


def _c_prototypes():
    """name -> (return kind, [arg kinds]) from include/swb200.h; kinds: 'int' (32-bit), 'long' (64-bit), 'ptr', 'void'."""
    with open(os.path.join(ROOT, "include", "swb200.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    text = re.sub(r"#.*", "", text)

    def kind(t):
        t = t.strip()
        if "*" in t:
            return "ptr"
        base = t.replace("const", "").split()
        if not base or base == ["void"]:
            return "void"
        if base[0] in ("int64_t", "uint64_t"):
            return "long"
        assert base[0] in ("int", "int32_t", "uint32_t"), t
        return "int"

    out = {}
    for m in re.finditer(r"([A-Za-z_][A-Za-z0-9_ \*]*?)\b(swb_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        arglist = [a for a in (x.strip() for x in args.split(",")) if a and a != "void"]
        # drop the parameter name: everything up to the last identifier
        kinds = [kind(re.sub(r"\b[A-Za-z_][A-Za-z0-9_]*$", "", a) if not a.rstrip().endswith("*") else a) for a in arglist]
        out[name] = (kind(ret), kinds)
    return out


def test_ctypes_and_java_bindings_match_the_header():
    """No JDK exists here, so the Java layer cannot be compiled: at least its Panama descriptors (and the ctypes
    signatures the tests run through) must agree with swb200.h argument by argument."""
    import ctypes as C
    protos = _c_prototypes()
    assert len(protos) >= 30

    def ckind(t):
        if t is None:
            return "void"
        if t in (C.c_int, C.c_int32, C.c_uint32):
            return "int"
        if t in (C.c_int64, C.c_uint64, C.c_longlong):
            return "long"
        return "ptr"

    for name, (restype, argtypes) in _ffi.SIGNATURES.items():
        ret, args = protos[name]
        assert [ckind(a) for a in argtypes] == args, (name, args)
        assert ckind(restype) == ret, (name, ret)

    with open(os.path.join(ROOT, "java", "ffm", "sw", "NativeSW.java")) as f:
        java = f.read()
    jk = {"JAVA_INT": "int", "JAVA_LONG": "long", "ADDRESS": "ptr"}
    found = 0
    for m in re.finditer(r'h\(\s*"(swb_[a-z0-9_]+)"\s*,\s*FunctionDescriptor\.(ofVoid|of)\(([^)]*)\)', java):
        name, how, desc = m.group(1), m.group(2), [x.strip() for x in m.group(3).split(",") if x.strip()]
        ret, args = protos[name]
        kinds = [jk[d] for d in desc]
        if how == "of":
            assert kinds[0] == ret, (name, kinds[0], ret)
            kinds = kinds[1:]
        else:
            assert ret == "void", name
        assert kinds == args, (name, kinds, args)
        found += 1
    assert found >= 12


def test_jni_shim_compiles_and_matches_the_java_natives(tmp_path):
    """The JDK-8 host layer (java/sw/NativeSW.java) binds jni/swb_jni.c.  No JDK exists here: the shim is compiled
    against tests/jni_stub/jni.h and linked with libswb200; every `static native` method must have a
    Java_sw_NativeSW_<name> export whose C parameter list is (JNIEnv*, jclass, <one per Java argument>)."""
    import subprocess
    so = tmp_path / "libswbjni_stub.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "tests", "jni_stub"),
                           "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "jni", "swb_jni.c"),
                           "-L" + os.path.dirname(_ffi.LIB_PATH), "-lswb200", "-o", str(so)])
    exported = {l.split()[-1] for l in subprocess.check_output(["nm", "-D", "--defined-only", str(so)], text=True).splitlines()
                if "Java_sw_NativeSW_" in l}
    with open(os.path.join(ROOT, "java", "sw", "NativeSW.java")) as f:
        java = f.read()
    natives = re.findall(r"static\s+native\s+[\w\[\]]+\s+(\w+)\s*\(([^)]*)\)\s*;", java)
    assert len(natives) >= 25
    with open(os.path.join(ROOT, "jni", "swb_jni.c")) as f:
        csrc = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    for name, args in natives:
        sym = "Java_sw_NativeSW_" + name
        assert sym in exported, sym
        m = re.search(sym + r"\s*\(([^)]*)\)", csrc)
        n_c = len([a for a in m.group(1).split(",") if a.strip()])
        n_java = len([a for a in args.split(",") if a.strip()])
        assert n_c == n_java + 2, (name, n_c, n_java)
    assert len(exported) == len(natives)
    # every swb_* symbol the shim calls is declared in the header (it compiled with -Werror) and exported by the library
    undefined = {l.split()[-1] for l in subprocess.check_output(["nm", "-D", "--undefined-only", str(so)], text=True).splitlines()
                 if " swb_" in l}
    lib_syms = {l.split()[-1] for l in subprocess.check_output(["nm", "-D", "--defined-only", _ffi.LIB_PATH], text=True).splitlines()}
    assert undefined and undefined <= lib_syms


def test_running_median_and_refset_info(tmp_path):
    """metrics.RunningMedian / RefSetInfo mirror the reference's reporter (src/metrics/RunningMedian.java:111-171,
    RefSetInfo.java:56-196): two-heap median, per-directory statistics, Java-formatted report."""
    import random
    import statistics
    from sparksmithwaterman_b200 import metrics
    rnd = random.Random(3)
    rm = metrics.RunningMedian()
    seen = []
    for _ in range(500):
        v = rnd.randint(0, 5000)
        seen.append(v)
        rm.add(v)
        assert rm.get_running_median() == statistics.median(seen)
    (tmp_path / "sub").mkdir()
    (tmp_path / "b.fa").write_text(">gi|1|x\nACGT\nAC\n>gi|2|y\nA\n")
    (tmp_path / "sub" / "a.fa").write_text(">gi|3|z\n" + "ACGTACGTAC" * 123 + "\n")
    d, n_files, longs, doubles, files = metrics.RefSetInfo.get_info(str(tmp_path))
    assert n_files == 2 and longs == [3, 1237, 1, 1230] and doubles[1] == 6.0 and abs(doubles[0] - 1237 / 3) < 1e-9
    assert sorted(files) == [("a.fa", 1), ("b.fa", 2)]
    text = metrics.RefSetInfo.all_info_str(str(tmp_path))
    assert "# reference sequences  =  3          \n" in text and "# total base pairs     =  1,237      \n" in text
    assert "max     =  1,230     \n" in text and "mean    =  412.33 \n" in text and "median  =  6.00   \n" in text
    assert "File Name                          |# Sequences\n-----------------------------------+-----------\n" \
           "a.fa                               |          1\nb.fa                               |          2\n" in text
    assert metrics.info_of_lengths([])[0] == [0, 0, (1 << 63) - 1, 0]


def test_rows_per_lane_classes_cover_the_short_path():
    """swb_internal.h: every read length of the s16x2 path (1 .. MAX_LONG_ROWS) has a rows-per-lane class with
    8 * K >= m, the class list is ascending, the classes above MAX_K_BASE (biased fill + tile kernels only) reach
    MAX_LONG_ROWS, and the row index of a max-cell key (KEY_I_BITS) can hold it.  Each launcher's switch lists the
    classes it is compiled for."""
    import re
    src = open(os.path.join(ROOT, "sparksmithwaterman_b200", "csrc", "swb_internal.h")).read()
    gl = int(re.search(r"constexpr int GL = (\d+);", src).group(1))
    body = re.search(r"kKList\[kNumK\] = \{([^}]*)\}", src, re.S).group(1)
    ks = [int(x) for x in re.sub(r"//[^\n]*", "", body).replace("\n", " ").split(",") if x.strip()]
    n = int(re.search(r"constexpr int kNumK = (\d+);", src).group(1))
    assert len(ks) == n and ks == sorted(ks)
    k_base = int(re.search(r"constexpr int MAX_K_BASE = (\d+);", src).group(1))
    long_rows = int(re.search(r"constexpr int MAX_LONG_ROWS = (\d+);", src).group(1))
    i_bits = int(re.search(r"KEY_I_BITS = (\d+)", src).group(1))
    assert gl * k_base == 256 and gl * ks[-1] >= long_rows and long_rows < (1 << i_bits)
    for m in range(1, long_rows + 1):
        k = next(k for k in ks if gl * k >= m)
        assert gl * k - m < max(gl * 8, m // 4 + gl), (m, k)        # padding stays small
    csrc = os.path.join(ROOT, "sparksmithwaterman_b200", "csrc")
    for fname, fn, wanted in (("swb_fill_bias.cu", "launch_fill_bias_k", ks), ("swb_trace_tile.cu", "launch_tile_trace_k", ks),
                              ("swb_trace_tile.cu", "launch_tile_locate_k", ks), ("swb_fill.cu", "launch_fill_k", [k for k in ks if k <= k_base]),
                              ("swb_trace.cu", "launch_trace_k", [k for k in ks if k <= k_base])):
        text = open(os.path.join(csrc, fname)).read()
        got = sorted(int(x) for x in re.findall(r"case (\d+):\s+return " + fn + r"<\1>", text))
        assert got == wanted, (fname, fn, got)


def test_library_reads_only_documented_environment_variables():
    """Every kernel and launch shape follows from the inputs: the library reads only the two variables INTEGRATION.md
    documents, SWB_NCCL_LIB (where NCCL is) and SWB_QUEUE_LINGER_US (how long the submission queue waits for more
    pairs), neither of which selects an implementation."""
    csrc = os.path.join(ROOT, "sparksmithwaterman_b200", "csrc")
    names = set()
    for fname in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, fname)) as f:
            names.update(re.findall(r"getenv\s*\(\s*([^)]*?)\s*\)", f.read()))
    assert names == {'"SWB_NCCL_LIB"', '"SWB_QUEUE_LINGER_US"'}, names
