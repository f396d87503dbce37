"""CPU-side checks (run with -m "not gpu"): the C-ABI library builds, loads and exports every
symbol include/deeprec_b200.h declares; host-side argument validation rejects bad calls before
any launch; the product path refuses to run without CUDA (no CPU fallback)."""
import ctypes

import numpy as np
import pytest
import torch


def test_library_exports_every_header_symbol():
    from deep_recommenders_b200 import _lib, build
    build.build()
    lib = _lib.load()
    names = _lib.header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/deeprec_b200.h but not exported"
    assert set(names) == set(_lib._SIGS), "ctypes signature table out of sync with the header"
    assert lib.dr_version() == 100


def test_host_side_validation_without_gpu():
    from deep_recommenders_b200 import _lib
    lib = _lib.load()
    # D not a multiple of 4 -> DR_EINVAL before any CUDA call
    rc = lib.dr_gather_fwd(16, 10, 16, 8, 4, 6, 16, None)
    assert rc == -1 and b"D=6" in lib.dr_last_error()
    rc = lib.dr_gather_fwd(None, 10, 16, 8, 4, 16, 16, None)
    assert rc == -1
    rc = lib.dr_gather_fwd(8, 10, 16, 8, 4, 16, 16, None)          # misaligned table base
    assert rc == -2
    rc = lib.dr_dense_fwd(16, 16, None, 4, 0, 3, 0, 16, None)
    assert rc == -1
    rc = lib.dr_cross_fwd(16, 16, 16, None, None, None, -1.0, 4, 8, 0, None, 16, 16, None)
    assert rc == -1 and b"non-negative" in lib.dr_last_error()
    rc = lib.dr_inbatch_softmax_fwd(16, 16, None, None, None, 1.0, 4, 4, 6, 16, 16, None)
    assert rc == -1
    assert lib.dr_tune_set(b"no_such_knob", 1) == -1
    with pytest.raises(ValueError):
        _lib.check(-1, "x")


def test_no_cpu_fallback():
    from deep_recommenders_b200 import ops
    from deep_recommenders_b200._lib import DeepRecError
    with pytest.raises(DeepRecError):
        ops.FMInteraction.apply(torch.randn(4, 3, 2))
    with pytest.raises(DeepRecError):
        ops.DenseFn.apply(torch.randn(4, 3), torch.randn(3, 2), None, 0)


def test_product_does_not_import_oracle():
    import pathlib
    root = pathlib.Path(__file__).resolve().parent.parent / "deep_recommenders_b200"
    for f in root.rglob("*.py"):
        text = f.read_text()
        assert "import oracle" not in text and "from oracle" not in text, f


def test_reference_import_paths():
    from deep_recommenders.keras.models.ranking import FM, FactorizationMachine, DeepFM   # noqa: F401
    from deep_recommenders.keras.models.ranking.dcn import Cross                          # noqa: F401
    from deep_recommenders.keras.models.retrieval import sbcnm                            # noqa: F401
    from deep_recommenders.estimator.models.feature_interaction import fm, FM as EFM, dnn  # noqa: F401
    c = Cross(projection_dim=None, diag_scale=0.1)
    cfg = c.get_config()
    for k in ("projection_dim", "diag_scale", "use_bias", "kernel_init", "kernel_regu", "bias_init", "bias_regu"):
        assert k in cfg
    assert cfg["kernel_init"]["class_name"] == "TruncatedNormal"
    with pytest.raises(AssertionError):
        Cross(diag_scale=-0.5)


def test_hashing_known_answers():
    from deep_recommenders_b200.hashing import fingerprint64, hash_bucket
    assert fingerprint64(b"") == 0x9AE16A3B2F90404F
    assert fingerprint64(b"abc") == 2640714258260161385          # pyfarmhash README
    assert fingerprint64(b"hello") == 13009744463427800296
    # tf.strings.to_hash_bucket_fast(["Hello", "TensorFlow", "2.x"], 3) -> [0, 2, 2] (TF API docs)
    assert hash_bucket(["Hello", "TensorFlow", "2.x"], 3).tolist() == [0, 2, 2]
    assert hash_bucket([1, "1", b"1"], 100).tolist()[0] == hash_bucket(["1"], 100)[0]


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` runs without a GPU and prints the contract's JSON line."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "examples/s" and line["value"] > 0
    assert line["metric"].startswith("examples/sec (fwd+bwd) DeepFM")
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True


def test_bench_dump_outputs_writes_float32_arrays_of_a_fixed_row_sample(tmp_path, monkeypatch):
    """`bench.py --dump-outputs DIR` (on a stand-in trainer over CPU tensors): every array is a float32 .npy, two dumps of
    the same state are identical, and the embedding sample holds distinct table rows in ascending order with their own
    first-order weights."""
    import os
    import types
    import bench
    from deep_recommenders_b200.embedding import EmbeddingCollection
    coll = EmbeddingCollection([1000, 2000, 500], 16, device="cpu", seed=1)
    with torch.no_grad():
        coll.lin_view().copy_(torch.arange(coll.total_rows, dtype=torch.float32))
    trainer = types.SimpleNamespace(coll=coll, loss=torch.ones(1), prob=torch.rand(64), w=[torch.rand(48, 8), torch.rand(8, 1)],
                                    b=[torch.rand(8), None], flush_optimizer=lambda: None)
    monkeypatch.setattr(bench, "DUMP_EMBED_BYTES", 64 * 16 * 4)
    bench.dump_outputs(trainer, str(tmp_path / "a"))
    bench.dump_outputs(trainer, str(tmp_path / "b"))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["dense0_bias.npy", "dense0_kernel.npy", "dense1_kernel.npy", "embed_rows.npy", "fm_bias.npy",
                     "linear_rows.npy", "loss.npy", "prob.npy"]
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert a.dtype == np.float32 and np.array_equal(a, np.load(tmp_path / "b" / n)), n
    idx = np.load(tmp_path / "a" / "linear_rows.npy").astype(np.int64)
    assert len(idx) == 64 and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "embed_rows.npy"), coll.emb_view().detach().numpy()[idx])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "dense0_kernel.npy"), trainer.w[0].numpy())


def test_ctypes_signatures_match_the_header_arity_and_pointer_kinds():
    """Every entry of _lib._SIGS must have exactly the parameters its declaration in include/deeprec_b200.h has, with
    pointers bound as pointers, 64-bit integers as c_int64, ints as c_int and floats as c_float (an ABI drift here
    corrupts arguments silently at run time)."""
    import ctypes as C
    import re
    from deep_recommenders_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", _lib.HEADER_PATH.read_text(), flags=re.S)
    decls = {m.group(1): m.group(2) for m in re.finditer(r"\b(dr_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S)}
    assert set(decls) == set(_lib._SIGS)
    for name, params in decls.items():
        plist = [p.strip() for p in params.split(",")] if params.strip() not in ("", "void") else []
        sig = _lib._SIGS[name]
        assert len(plist) == len(sig), f"{name}: header has {len(plist)} parameters, ctypes table {len(sig)}"
        for p, ct in zip(plist, sig):
            if "*" in p:
                assert ct in (C.c_void_p, C.c_char_p), f"{name}: '{p}' must be bound as a pointer, got {ct}"
            elif re.match(r"(const\s+)?(int64_t|uint64_t)\b", p):
                assert ct in (C.c_int64, C.c_uint64), f"{name}: '{p}' must be 64-bit, got {ct}"
            elif re.match(r"(const\s+)?float\b", p):
                assert ct is C.c_float, f"{name}: '{p}' must be c_float, got {ct}"
            elif re.match(r"(const\s+)?int\b", p):
                assert ct is C.c_int, f"{name}: '{p}' must be c_int, got {ct}"
            else:
                raise AssertionError(f"{name}: unclassified parameter '{p}'")


def test_every_call_site_passes_the_declared_number_of_arguments():
    """Static check of all `lib.dr_*(...)` call sites in the package, tests and tools (GPU-only code paths cannot run
    here; a wrong argument count would only surface on the GPU box)."""
    import ast
    import pathlib
    from deep_recommenders_b200 import _lib
    root = pathlib.Path(__file__).resolve().parent.parent
    files = list((root / "deep_recommenders_b200").rglob("*.py")) + list((root / "tests").glob("*.py")) + \
        list((root / "tools").glob("*.py")) + [root / "bench.py", root / "__graft_entry__.py"]
    checked = 0
    for f in files:
        for node in ast.walk(ast.parse(f.read_text())):
            if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr in _lib._SIGS:
                if any(isinstance(a, ast.Starred) for a in node.args) or node.keywords:
                    continue
                want = len(_lib._SIGS[node.func.attr])
                assert len(node.args) == want, f"{f.name}:{node.lineno}: {node.func.attr} called with {len(node.args)} " \
                                               f"arguments, the C-ABI takes {want}"
                checked += 1
    assert checked > 60


def test_plain_c_program_links_and_calls_the_library(tmp_path):
    """The boundary is a C ABI: a C99 program compiled with gcc against include/deeprec_b200.h links to the .so and
    gets the same answers as the Python binding (host entry points only; no GPU, no torch, no Python)."""
    import pathlib
    import shutil
    import subprocess
    from deep_recommenders_b200 import _lib
    from deep_recommenders_b200.hashing import hash_bucket
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    root = pathlib.Path(__file__).resolve().parent.parent
    libdir = _lib.LIB_PATH.parent
    exe = tmp_path / "c_abi_host_demo"
    cmd = [gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", str(root / "include"),
           str(root / "examples" / "c_abi_host_demo.c"), "-L", str(libdir), "-ldeeprec_b200",
           f"-Wl,-rpath,{libdir}", "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.strip().splitlines()
    assert lines[0] == "version 100"
    assert lines[1] == "to_hash_bucket_fast 0 2 2"                       # TF API docs example
    assert lines[2] == "fingerprint64(abc) 2640714258260161385"
    assert lines[3] == "crc32c(123456789) e3069283"
    want = hash_bucket(np.array([6040, -1], dtype=np.int64), 1000).tolist()
    assert lines[4] == f"hash_bucket_i64 {want[0]} {want[1]}"
    assert lines[5].startswith("dr_gather_fwd(D=6) rc=-1") and "D=6" in lines[5]


def test_shipped_library_contains_the_blackwell_kernels_it_claims():
    """Static check of the built .so (no GPU): the CTA-pair tcgen05 GEMM and the single-CTA one are in it, sized to be
    launchable (no spills to local memory, registers x threads within the SM's file), and the pair kernel really is a
    cta_group::2 kernel (UTCHMMA.2CTA, the multicast commit, the cluster barrier) fed by TMA."""
    import os
    import re
    import shutil
    import subprocess
    from deep_recommenders_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not installed")
    _lib.load()
    so = str(_lib.LIB_PATH)
    res = subprocess.run([cuobjdump, "-res-usage", so], capture_output=True, text=True, check=True).stdout.splitlines()
    found = {}
    for i, line in enumerate(res):
        m = re.match(r"\s*Function (\S+):", line)
        if m and i + 1 < len(res):
            r = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", res[i + 1])
            if r:
                found[m.group(1)] = tuple(map(int, r.groups()))
    pair = {k: v for k, v in found.items() if "gemm_tc_pair_kernel" in k}
    single = {k: v for k, v in found.items() if "14gemm_tc_kernel" in k}
    assert len(pair) == 8 and len(single) >= 16, (len(pair), len(single))
    for k, (reg, stack, shared, local) in pair.items():
        assert local == 0 and stack == 0 and reg * 320 <= 65536, (k, reg, stack, local)
    name = next(k for k in pair if "ILi256ELi3ELb0ELb1E" in k)          # the forward instantiation of the C2 / C5 towers
    sass = subprocess.run([cuobjdump, "-sass", "-fun", name, so], capture_output=True, text=True, check=True).stdout
    for op in ("UTCHMMA.2CTA", "UTCBAR.2CTA.MULTICAST", "UCGABAR_ARV", "UTMALDG.2D", "UTMASTG.2D", "UTMAREDG.2D.ADD", "LDTM"):
        assert op in sass, f"{op} missing from {name}"
