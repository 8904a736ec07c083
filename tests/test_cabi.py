"""The C-ABI library builds here (nvcc cross-compiles without a GPU), loads, and exports every symbol that
include/esf.h declares.  No compute calls: those are in the -m gpu tests."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    src = open(os.path.join(ROOT, "include", "esf.h")).read()
    return re.sub(r"/\*.*?\*/", "", src, flags=re.S)


def _declared_symbols():
    return sorted(set(re.findall(r"\b(esf_[a-z0-9_]+)\s*\(", _header())))


def _declarations():
    """{name: (return type, [(parameter type, parameter name)])} of every function include/esf.h declares."""
    decls = {}
    for ret, name, params in re.findall(r"((?:const\s+)?\w+\s*\**)\s*\b(esf_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", _header()):
        args = []
        for p in params.split(","):
            p = " ".join(p.split())
            if p and p != "void":
                ctype, pname = re.match(r"(.*?)\s*(\w+)$", p).groups()
                args.append((ctype, pname))
        decls[name] = (ret.replace(" ", ""), args)
    return decls


def _ctypes_of(ctype, pname):
    """The ctypes type the binding must give a parameter of C type `ctype`."""
    from efficient_slowfast_b200 import runtime as rt

    base = ctype.replace("const", "").replace(" ", "")
    if base == "esf_view*":
        return ctypes.POINTER(rt.EsfView)
    if base == "esf_conv_desc*":
        return ctypes.POINTER(rt.EsfConvDesc)
    if base == "esf_op**":
        return ctypes.POINTER(ctypes.c_void_p)
    # int32_t* out-parameters and the host int32 tables (esf.h: a name ending in _host, and chan_src "host int32[C]")
    if base == "int32_t*" and ("const" not in ctype or pname.endswith("_host") or pname == "chan_src"):
        return ctypes.POINTER(ctypes.c_int32)
    if base.endswith("*"):
        return ctypes.c_void_p       # device pointers, esf_op*, the stream
    return {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}[base]


def test_header_symbols_exported(esf_lib):
    syms = _declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(esf_lib, s), "libesf_b200.so does not export %s" % s
    assert esf_lib.esf_version() >= 100


def test_binding_signatures_match_header(esf_lib):
    """runtime.lib()'s argtypes / restype are the Python side's only description of the C ABI, and Plan._bind converts
    arguments by them: every function include/esf.h declares has its parameters' kinds, in order."""
    decls = _declarations()
    assert set(decls) == set(_declared_symbols())
    restypes = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "constchar*": ctypes.c_char_p, "void": None}
    for name, (ret, params) in sorted(decls.items()):
        f = getattr(esf_lib, name)
        assert f.restype is restypes[ret], "%s returns %s, bound as %s" % (name, ret, f.restype)
        if not params and f.argtypes is None:
            continue
        assert f.argtypes is not None, "%s has no argtypes" % name
        assert len(f.argtypes) == len(params), "%s: %d argtypes for %d parameters" % (name, len(f.argtypes), len(params))
        for i, ((ctype, pname), got) in enumerate(zip(params, f.argtypes)):
            want = _ctypes_of(ctype, pname)
            assert got is want, "%s parameter %d (%s %s): bound as %s, expected %s" % (name, i, ctype, pname, got, want)


def test_geometry_rule(esf_lib):
    from efficient_slowfast_b200 import runtime as rt

    assert rt.igemm_geometry(64, 256) == (64, 1, 256, 256)
    assert rt.igemm_geometry(72, 64) == (64, 2, 64, 64)
    assert rt.igemm_geometry(8, 32) == (16, 1, 32, 32)
    assert rt.igemm_geometry(32, 8) == (32, 1, 16, 16)
    assert rt.igemm_geometry(1152, 2048) == (64, 18, 256, 2048)


def test_bad_sizes_and_null_descriptors_give_error_codes(esf_lib):
    from efficient_slowfast_b200 import runtime as rt

    assert esf_lib.esf_igemm_geometry(0, 4, None, None, None, None) < 0
    assert b"positive" in esf_lib.esf_last_error()
    assert esf_lib.esf_attn_tc_pack_bytes(2, 100, 0) < 0
    assert esf_lib.esf_attn_tc_pack_bytes(2, 100, 129) < 0    # d > 128 is the CUDA-core fallback's (esf_attn_generic)
    assert esf_lib.esf_attn_tc_pack_bytes(2, 100, 8) > 0
    h = ctypes.c_void_p()
    assert esf_lib.esf_conv_igemm_create(None, ctypes.byref(h)) < 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_forward_without_gpu_fails_loudly():
    """No CPU fallback: the drop-in model refuses CPU tensors instead of silently computing elsewhere."""
    import efficient_slowfast_b200 as esf
    from efficient_slowfast_b200 import runtime as rt

    cfg = esf.slowfast_dual_8x8_r50_cfg()
    cfg.NUM_GPUS = 0
    m = esf.build_model(cfg).eval()
    with pytest.raises(rt.EsfError):
        m([torch.zeros(1, 3, 8, 32, 32), torch.zeros(1, 3, 32, 32, 32)])
    m.train()
    with pytest.raises(NotImplementedError):
        m([torch.zeros(1, 3, 8, 32, 32), torch.zeros(1, 3, 32, 32, 32)])


def test_production_kernels_keep_their_resource_budget(esf_lib):
    """Guard for a regression measured in round 2: adding run-time flags to the position-attention kernel changed the
    register allocation of its default instantiation (96 -> 88) and cost 4-6 % of the step although the flags were off
    (profiles/r2_attention_experiments.md section 5).  The library holds exactly the production instantiations of the
    hot kernels (no experiment variants), and they keep the resources they were tuned with and use no local memory."""
    import shutil
    import subprocess

    from efficient_slowfast_b200 import runtime

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-res-usage", runtime.lib_path()], stdout=subprocess.PIPE, text=True).stdout
    usage = {}
    name = None
    for line in out.splitlines():
        line = line.strip()
        if line.startswith("Function "):
            name = line[len("Function "):].rstrip(":")
        elif line.startswith("REG:") and name:
            usage[name] = dict(kv.split(":") for kv in line.split() if ":" in kv and not kv.startswith("CONSTANT"))
    v2 = {n: u for n, u in usage.items() if "attn_tc_v2_kernel" in n}
    assert sorted(v2) == ["_ZN3esf17attn_tc_v2_kernelILb%dEEEvNS_12AttnTcParamsE" % f for f in (0, 1)], sorted(v2)
    for u in v2.values():   # 640 threads per CTA cap the kernel at 102 registers; the tuned loop uses 96
        assert int(u["REG"]) == 96 and int(u["LOCAL"]) == 0, u
    ig = [u for n, u in usage.items() if "igemm_kernel" in n]
    assert ig and all(int(u["REG"]) <= 104 and int(u["LOCAL"]) == 0 for u in ig), ig
    # the temporal-band stem's issuing warp is a serial instruction stream: no local memory, and one instantiation per
    # (k-steps 1..4, 16-bit format)
    tb = {n: u for n, u in usage.items() if "stem_tband_kernel" in n}
    assert len(tb) == 8 and all(re.search(r"stem_tband_kernelILi[1-4]ELb[01]EEEvNS_12StemTbParamsE$", n) for n in tb), sorted(tb)
    assert all(int(u["LOCAL"]) == 0 for u in tb.values()), tb


def test_library_reads_no_environment():
    """What a kernel computes and which kernel runs is a function of the call's arguments: an environment variable
    inherited on a shared machine must not switch the library to another code path (nothing in a log would show it)."""
    csrc = os.path.join(ROOT, "efficient_slowfast_b200", "csrc")
    hits = []
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            for i, line in enumerate(open(os.path.join(csrc, f)), 1):
                if re.search(r"\bgetenv\s*\(", line):
                    hits.append("%s:%d: %s" % (f, i, line.strip()))
    assert not hits, hits


def test_package_reads_no_environment():
    """The same rule one layer up: the plan builder picks kernels from shapes and parameters only.  The two exceptions
    read no switch: _build.py takes the compiler and its extra flags (NVCC, ESF_NVCC_EXTRA; the flags are part of the
    library's digest), workloads.py the directory test fixtures are read from (ESF_GOLDEN_DIR)."""
    pkg = os.path.join(ROOT, "efficient_slowfast_b200")
    hits = []
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".py") and f not in ("_build.py", "workloads.py"):
            for i, line in enumerate(open(os.path.join(pkg, f)), 1):
                if re.search(r"\b(environ|getenv)\b", line):
                    hits.append("%s:%d: %s" % (f, i, line.strip()))
    assert not hits, hits
