"""CPU: the C-ABI library loads and exports every symbol include/qpskcuda.h declares; the host-side
designers agree with the oracle; without a GPU every compute entry point fails loudly (no fallback).
No GPU compute calls are made here.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "qpskcuda.h")


def _declared_in_header():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"QPSK_API\s+[\w\s\*]+?\b(qpsk_\w+)\s*\(", text)))


def test_header_compiles_as_c():
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", HEADER])


def test_library_exports_every_declared_symbol(qp):
    names = _declared_in_header()
    assert len(names) >= 70
    lib = qp._native.lib()
    for n in names:
        assert hasattr(lib, n), f"libqpskcuda.so does not export {n}"
    # and the ctypes table binds exactly the header's surface
    assert sorted(qp._native.declared_symbols()) == names
    exported = subprocess.check_output(["nm", "-D", "--defined-only", qp._native.LIB_PATH], text=True)
    exported = sorted(set(re.findall(r"\bT (qpsk_\w+)", exported)))
    assert exported == names, set(exported) ^ set(names)      # nothing else leaks out of the library


def test_sass_is_sm100a_with_bulk_copies_and_ffma2(qp):
    sass = subprocess.check_output(["cuobjdump", "-sass", qp._native.LIB_PATH], text=True)
    assert "sm_100a" in sass
    assert "UBLKCP" in sass            # TMA bulk copies (cp.async.bulk) in the FIR kernel
    assert "FFMA2" in sass             # packed fp32x2 FMA
    assert "SYNCS" in sass             # mbarrier
    funcs = sass.split("Function : ")
    # kernels that restate the reference's unfused fp32 arithmetic must not contain fused multiply-adds
    for prefix in ("_ZN4qpsk18fir_generic_kernelILb1EE", "_ZN4qpsk9mm_kernel", "_ZN4qpsk13decode_kernel"):
        body = [f for f in funcs if f.startswith(prefix)]
        assert body, prefix
        assert " FFMA " not in body[0] and "FFMA2" not in body[0], prefix


def test_status_strings_and_version(qp):
    lib = qp._native.lib()
    assert lib.qpsk_version() >= 100
    for st in range(0, -9, -1):
        assert lib.qpsk_strerror(st)


def test_host_side_designers_match_oracle(qp, orc):
    for span, beta, fs, rs in [(10, float(np.float32(0.4)), 10_000_000, 5_000_000), (16, 0.35, 16000, 1000), (4, 0.25, 8000, 1000),
                               (6, 0.35, 2500, 1000), (11, 0.9, 10_000_000, 333333)]:
        assert np.array_equal(qp.RRCFilter.generateCoefficents(span, beta, fs, rs), orc.RRCFilter.generateCoefficents(span, beta, fs, rs))
    for sps, ro, n in [(2.0, 0.4, 40), (30.0, 0.9, 10), (4.0, 0.35, 13)]:
        lo, up = qp.fll_design(sps, ro, n)
        wlo, wup = orc.FLLBandEdgeFilter(sps, ro, n, 0.01).taps()
        assert np.array_equal(lo, wlo) and np.array_equal(up, wup)
    assert qp.mm_gains_from_bw(1e-4) == orc.mm_gains_from_bw(1e-4)
    n = C.c_int(0)
    assert qp._native.lib().qpsk_rrc_taps(6.0, 0.35, 4000, 1000, None, 0, C.byref(n)) == 0 and n.value == 25
    buf = (C.c_double * 4)()
    assert qp._native.lib().qpsk_rrc_taps(6.0, 0.35, 4000, 1000, buf, 4, C.byref(n)) == qp._native.ERR_CAPACITY


def test_no_cpu_fallback_without_device(qp):
    if qp.device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(qp.QpskCudaError):
        qp.ComplexFIRFilter(np.ones(4, np.float32))
    with pytest.raises(qp.QpskCudaError):
        qp.QPSKModulator(4000, 1000)
    with pytest.raises(qp.QpskCudaError):
        qp.QPSKDeModulator(4000, 1000)
    with pytest.raises(qp.QpskCudaError):
        qp.FLLBandEdgeFilter(4.0, 0.35, 40, 0.01)
    # argument validation still mirrors the reference before any device work
    with pytest.raises(qp.ArgumentException):
        qp.ComplexFIRFilter(np.ones(3, np.float32))
    with pytest.raises(qp.ArgumentNullException):
        qp.ComplexFIRFilter(None)


def test_product_never_references_the_oracle():
    """The oracle is test infrastructure: nothing under the package (or the built library) may touch it."""
    pkg = os.path.join(ROOT, "qpsk_modulator_demodulator_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in text and "from oracle" not in text and "liboracle" not in text, f
    needed = subprocess.check_output(["readelf", "-d", os.path.join(pkg, "lib", "libqpskcuda.so")], text=True)
    assert "oracle" not in needed


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` runs without a GPU (the CPU arm the driver times next to ours) and prints one JSON
    line with the contract's keys; under torchrun only rank 0 prints."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Msamples/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["metric"].startswith("Msamples/s RRC FIR")
    r1 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=600, env=dict(env, RANK="1", WORLD_SIZE="2"), cwd=root)
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_csharp_bindings_match_the_header():
    """integration/csharp cannot be compiled here (no .NET): at least every P/Invoke it declares must name an entry point
    of include/qpskcuda.h with the same number of parameters, and the shim must only call bindings that exist."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "qpskcuda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    protos = {}
    for m in re.finditer(r"QPSK_API\s+[\w\s\*]+?\b(qpsk_\w+)\s*\(([^;]*?)\)\s*;", hdr, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    native = open(os.path.join(root, "integration", "csharp", "QpskCuda.Native.cs")).read()
    native = re.sub(r"//[^\n]*", " ", native)
    bound = {}
    for m in re.finditer(r"static\s+extern\s+\w+\s+(qpsk_\w+)\s*\(([^;]*?)\)\s*;", native, flags=re.S):
        args = m.group(2).strip()
        bound[m.group(1)] = 0 if args == "" else len(args.split(","))
    assert len(bound) >= 30
    for name, n in bound.items():
        assert name in protos, f"{name} is not declared in qpskcuda.h"
        assert n == protos[name], f"{name}: {n} parameters in C#, {protos[name]} in the header"
    # parameter by parameter: the C# type must marshal as the C type (int64_t <-> long, T* <-> T* / out T / in T,
    # handles <-> IntPtr, handle out-parameters <-> out IntPtr, const char* <-> byte* / string)
    ok_map = {
        "int": [("", "int")], "int64_t": [("", "long")], "float": [("", "float")], "double": [("", "double")],
        "float*": [("", "float*"), ("out", "float"), ("in", "float")], "double*": [("", "double*"), ("out", "double")],
        "int*": [("", "int*"), ("out", "int")], "int64_t*": [("", "long*"), ("out", "long")],
        "uint8_t*": [("", "byte*")], "char*": [("", "byte*"), ("", "string?"), ("", "string")], "void*": [("", "IntPtr"), ("", "void*")],
    }
    cargs = {}
    for m in re.finditer(r"QPSK_API\s+[\w\s\*]+?\b(qpsk_\w+)\s*\(([^;]*?)\)\s*;", hdr, flags=re.S):
        a = m.group(2).strip()
        cargs[m.group(1)] = [] if a in ("", "void") else [v.strip() for v in a.split(",")]
    for m in re.finditer(r"static\s+extern\s+\w+\s+(qpsk_\w+)\s*\(([^;]*?)\)\s*;", native, flags=re.S):
        for ca, sa in zip(cargs[m.group(1)], [v for v in m.group(2).split(",") if v.strip()]):
            ct = re.sub(r"\s+", " ", re.sub(r"\bconst\b", "", ca)).strip()
            ct = re.match(r"(.*?)(\w+)$", ct).group(1).strip().replace(" *", "*")
            mm = re.match(r"(?:(out|in|ref)\s+)?([\w\?\*]+)\s+\w+$", sa.strip())
            got = (mm.group(1) or "", mm.group(2))
            if re.match(r"qpsk_\w+\*\*$", ct):
                good = got == ("out", "IntPtr")
            elif re.match(r"qpsk_\w+\*$", ct):
                good = got == ("", "IntPtr")
            else:
                good = got in ok_map.get(ct, [])
            assert good, f"{m.group(1)}: C `{ca}` against C# `{sa.strip()}`"
    shim = open(os.path.join(root, "integration", "csharp", "QpskCuda.Shim.cs")).read()
    used = set(re.findall(r"QpskCuda\.(qpsk_\w+)\s*\(", shim))
    assert used and used <= set(bound), sorted(used - set(bound))


# ---------------------------------------------------------------------------------------------------------------------
# what the C# shim RETURNS (round-1 review: three span overloads returned float counts where the reference returns complex
# counts).  The shim cannot be compiled here, so its method bodies are parsed and every value-returning member on the path
# is checked against a table of the reference's conventions; the table itself is checked against the reference's own
# source text of the same members when QPSK_REFERENCE_DIR names the reference's Modulation-Simulation directory.
# ---------------------------------------------------------------------------------------------------------------------
def _cs_strip(text):
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    return re.sub(r"//[^\n]*", " ", text)


def _cs_method_body(text, cls, sig_regex):
    """Body (between the outer braces) of the first member of class `cls` whose signature matches `sig_regex`."""
    m = re.search(r"\bclass\s+" + re.escape(cls) + r"\b", text)
    assert m, cls
    i = text.index("{", m.end())
    depth, j = 0, i
    while True:                      # class extent
        if text[j] == "{":
            depth += 1
        elif text[j] == "}":
            depth -= 1
            if depth == 0:
                break
        j += 1
    body = text[i:j]
    m = re.search(sig_regex, body)
    assert m, (cls, sig_regex)
    i = body.index("{", m.end())
    depth, j = 0, i
    while True:
        if body[j] == "{":
            depth += 1
        elif body[j] == "}":
            depth -= 1
            if depth == 0:
                break
        j += 1
    return body[i + 1:j]


def _cs_last_return(body):
    r = re.findall(r"\breturn\s+([^;]+);", body)
    assert r, body
    return re.sub(r"\s+", "", r[-1])


def _cs_resolve(body, expr):
    """`return n;` -> the initialiser of `int n = ...;` in the same body (one level)."""
    m = re.search(r"\bint\s+" + re.escape(expr) + r"\s*=\s*([^;]+);", body)
    return re.sub(r"\s+", "", m.group(1)) if m else expr


SPAN2 = r"\(\s*ReadOnlySpan<float>\s+(\w+)\s*,\s*Span<float>\s+(\w+)\s*\)"
# (class, reference file, signature, expected return as a function of the first parameter name `x`)
RETURNS = [
    ("FLLBandEdgeFilter", "Models/Band-Edge Filter.cs", r"public\s+int\s+Process" + SPAN2, "{x}.Length>>1"),
    ("CostasLoopQpsk", "Models/CostasLoopQpsk.cs", r"public\s+int\s+Process" + SPAN2, "{x}.Length>>1"),
    ("MuellerMuller", "Models/MuellerMuller.cs", r"public\s+int\s+Process" + SPAN2, "<symbols>"),
]


def test_csharp_shim_return_values_follow_the_reference():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    shim = _cs_strip(open(os.path.join(root, "integration", "csharp", "QpskCuda.Shim.cs")).read())
    for cls, _, sig, want in RETURNS:
        body = _cs_method_body(shim, cls, sig)
        x = re.search(sig, shim[shim.index("class " + cls):]).group(1)
        got = _cs_resolve(body, _cs_last_return(body))
        if want == "<symbols>":
            # the count the native call reports in its `out int nSym` (complex symbols), unscaled
            m = re.search(r"qpsk_mm_process\s*\([^;]*out\s+(\w+)\s*\)", body)
            assert m and got == m.group(1), (cls, got)
        else:
            assert got == want.format(x=x), (cls, got)
    # allocating overloads: array sizes in floats = 2 x complex count (MuellerMuller.cs:148-156, QPSKDeModulator.cs:446)
    mm = re.sub(r"\s+", "", _cs_method_body(shim, "MuellerMuller", r"public\s+float\[\]\s+Process\s*\(\s*float\[\]"))
    assert "newfloat[maxSymbols<<1]" in mm and "newfloat[n<<1]" in mm and "if(n==maxSymbols)returntmp;" in mm
    con = re.sub(r"\s+", "", _cs_method_body(shim, "QPSKDeModulator", r"public\s+float\[\]\s+deModulateConstellation"))
    assert "newfloat[nSym<<1]" in con


def test_reference_source_has_the_conventions_the_shim_follows():
    """The conventions table above against the reference's own C# source.  Those sources are not part of this repository:
    set QPSK_REFERENCE_DIR to the reference's Modulation-Simulation directory to run this comparison."""
    ref_root = os.environ.get("QPSK_REFERENCE_DIR")
    if not ref_root:
        pytest.skip("QPSK_REFERENCE_DIR is not set: the reference's C# sources are not part of this repository")
    assert os.path.isdir(ref_root), f"QPSK_REFERENCE_DIR={ref_root} is not a directory"
    for cls, ref_file, sig, want in RETURNS:
        ref = _cs_strip(open(os.path.join(ref_root, ref_file), errors="replace").read())
        rbody = _cs_method_body(ref, cls, sig)
        rx = re.search(sig, ref[ref.index("class " + cls):]).group(1)
        rgot = _cs_last_return(rbody) if want == "<symbols>" else _cs_resolve(rbody, _cs_last_return(rbody))
        if want == "<symbols>":
            assert rgot == "outSymbols" and re.search(r"outSymbols\+\+", re.sub(r"\s+", "", rbody)), rgot
        else:
            assert rgot == want.format(x=rx), (cls, rgot)
    rmm = re.sub(r"\s+", "", _cs_method_body(_cs_strip(open(os.path.join(ref_root, "Models/MuellerMuller.cs")).read()),
                                             "MuellerMuller", r"public\s+float\[\]\s+Process\s*\(\s*float\[\]"))
    assert "newfloat[maxSymbols<<1]" in rmm and "newfloat[n<<1]" in rmm
    # the reference's callers use the MM count as a SYMBOL count: the demodulator loops k < nSymbols over 2-float steps
    # (QPSKDeModulator.cs:364-375); a shim returning floats would make them read twice too far
    dem = re.sub(r"\s+", "", _cs_strip(open(os.path.join(ref_root, "QPSKDeModulator.cs")).read()))
    assert "intnSymbols=symbolSync.Process(" in dem and "k<nSymbols" in dem


def test_csharp_shim_owns_handles_safely_and_checks_arguments_first():
    """ADVICE r1: handles must not leak when callers never Dispose (the reference classes are not IDisposable), and the
    reference's managed argument checks must run ahead of the native call with the reference's exception types."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    shim = _cs_strip(open(os.path.join(root, "integration", "csharp", "QpskCuda.Shim.cs")).read())
    assert re.search(r"class\s+QpskHandle\s*:\s*SafeHandle", shim) and "ReleaseHandle()" in shim
    for cls, destroy in [("ComplexFIRFilter", "qpsk_fir_destroy"), ("FLLBandEdgeFilter", "qpsk_fll_destroy"),
                         ("MuellerMuller", "qpsk_mm_destroy"), ("CostasLoopQpsk", "qpsk_costas_destroy"),
                         ("QPSKModulator", "qpsk_mod_destroy"), ("QPSKDeModulator", "qpsk_demod_destroy")]:
        seg = shim[shim.index("class " + cls):]
        seg = seg[:seg.index("public void Dispose()") + 60]
        assert "new QpskHandle(h, QpskCuda." + destroy + ")" in seg, cls
        assert "readonly IntPtr" not in seg, cls
    ctor = _cs_method_body(shim, "ComplexFIRFilter", r"public\s+ComplexFIRFilter\s*\(")
    flat = re.sub(r"\s+", "", ctor)
    # FIRFilter.cs:31-33: null -> ArgumentNullException; odd or EMPTY -> ArgumentException, before qpsk_fir_create
    assert flat.index("thrownewArgumentNullException") < flat.index("Length&1") < flat.index("Length==0") < flat.index("qpsk_fir_create")
    assert flat.count("thrownewArgumentException(") == 2
    mod = re.sub(r"\s+", "", _cs_method_body(shim, "QPSKModulator", r"public\s+float\[\]\s+ModulateTextUtf8"))
    assert mod.index("if(text==null)thrownewArgumentNullException(nameof(text))") < mod.index("ModulateBytes(")   # QPSKModulator.cs:81
    for cls, name in [("QPSKModulator", "ModulateBytes"), ("QPSKDeModulator", "DeModulateBytes")]:
        b = re.sub(r"\s+", "", _cs_method_body(shim, cls, r"public\s+\w+\[\]\s+" + name))
        assert b.index('startMarker.Length==0') < b.index('endMarker.Length==0') < b.index("QpskCuda.qpsk_"), (cls, name)
