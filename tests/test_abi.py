"""The C-ABI library loads and exports every symbol include/mcmc_gpu.h
declares (no compute calls: there is no GPU in the build container)."""
import ctypes as C

from mcmc_ocaml_b200 import _abi


def test_library_exports_every_declared_symbol():
    lib = _abi.load_library()
    declared = _abi.declared_symbols()
    assert len(declared) >= 50
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, f"missing symbols: {missing}"
    lib.mg_abi_version.restype = C.c_int
    assert lib.mg_abi_version() == 1


def test_struct_layouts_match_the_header():
    """sizes the C compiler gives the ABI structs (checked against gcc)"""
    import os
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    src = '#include <stdio.h>\n#include "mcmc_gpu.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",sizeof(mg_logfn),sizeof(mg_proposal),sizeof(mg_mcmc_cfg),sizeof(mg_into),sizeof(mg_rj_model),sizeof(mg_rjmcmc_cfg),sizeof(mg_nested_cfg));return 0;}'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(root, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        sizes = list(map(int, subprocess.check_output([os.path.join(d, "t")]).split()))
    want = [C.sizeof(x) for x in (_abi.mg_logfn, _abi.mg_proposal, _abi.mg_mcmc_cfg, _abi.mg_into, _abi.mg_rj_model,
                                  _abi.mg_rjmcmc_cfg, _abi.mg_nested_cfg)]
    assert sizes == want


def test_no_cpu_fallback():
    """without a CUDA device the product path must fail loudly"""
    import pytest
    import torch

    from mcmc_ocaml_b200 import Context, Failure
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(Failure):
        Context(0, 1)


def test_product_does_not_import_the_oracle():
    import os
    import re
    root = os.path.dirname(os.path.abspath(_abi.__file__))
    for dp, _, files in os.walk(root):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h")):
                text = open(os.path.join(dp, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle|#include\s+\"[^\"]*oracle/", text, re.M), f


def test_ocaml_stubs_parse_and_bind_existing_symbols():
    """No OCaml toolchain exists in this image, so ocaml/mcmc_gpu_stubs.c cannot be built.  It is at least parsed and
    type-checked by gcc against declaration-only mocks of <caml/*.h> (tests/c/caml_mock, shapes of the real runtime
    API), every `external` of mcmc_gpu.ml names a CAMLprim the C file defines, and every mg_* the stubs call is
    declared in include/mcmc_gpu.h."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    stubs = os.path.join(root, "ocaml", "mcmc_gpu_stubs.c")
    r = subprocess.run(["gcc", "-fsyntax-only", "-Wall", "-Werror=implicit-function-declaration", "-Werror=incompatible-pointer-types",
                        "-Wno-comment", "-I", os.path.join(root, "tests", "c", "caml_mock"), "-I", os.path.join(root, "include"), stubs],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    c_text = open(stubs).read()
    prims = set(re.findall(r"CAMLprim\s+value\s+(\w+)\s*\(", c_text))
    ml = open(os.path.join(root, "ocaml", "mcmc_gpu.ml")).read()
    externals = set(re.findall(r'"(mcmcgpu_\w+)"', ml))
    assert externals and externals <= prims, externals - prims
    called = set(re.findall(r"\b(mg_[a-z0-9_]+)\s*\(", c_text))
    assert called <= set(_abi.declared_symbols()), called - set(_abi.declared_symbols())
    # the .mli promises only what the .ml defines
    mli = open(os.path.join(root, "ocaml", "mcmc_gpu.mli")).read()
    for name in re.findall(r"^val\s+(\w+)", mli, re.M):
        assert re.search(r"^\s*(let|external)\s+(rec\s+)?" + name + r"\b", ml, re.M), name


def test_plugin_translation_unit_compiles_with_nvrtc():
    """The device headers embedded for run-time plugins (MH, RJMCMC and Nested kernels around a user log-density)
    compile with NVRTC for sm_100a -- no GPU needed for the compilation itself."""
    import ctypes
    import os
    import pytest
    try:
        nv = ctypes.CDLL("libnvrtc.so.12")
    except OSError:
        try:
            nv = ctypes.CDLL("/usr/local/cuda/lib64/libnvrtc.so.12")
        except OSError:
            pytest.skip("libnvrtc not present")
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    base = os.path.join(root, "mcmc_ocaml_b200", "csrc")
    names = ["rng.cuh", "models.cuh", "mcmc_kernel_dev.cuh", "kdtree.cuh", "rj_kernel_dev.cuh", "nested_kernel_dev.cuh",
             "../../include/mcmc_gpu.h"]
    srcs = [open(os.path.join(base, n)).read() for n in names]
    src = ("typedef signed char int8_t; typedef unsigned char uint8_t; typedef short int16_t; typedef unsigned short uint16_t;\n"
           "typedef int int32_t; typedef unsigned int uint32_t; typedef long long int64_t; typedef unsigned long long uint64_t;\n"
           "namespace mg_user { __device__ __forceinline__ double eval(int kind, const double *x, int dim, const double *p, long long np) {"
           " return -0.5 * x[0] * x[0]; } }\n"
           "#define MG_USER_EVAL(kind, x, d, p, np) mg_user::eval(kind, x, d, p, (long long)(np))\n"
           '#include "mcmc_kernel_dev.cuh"\n#include "rj_kernel_dev.cuh"\n#include "nested_kernel_dev.cuh"\n'
           'extern "C" __global__ void k_mh(const __grid_constant__ mg::MhArgs<mg::DynFn, mg::DynFn, mg::DynProp, 8> a) { mg::mh_ensemble_body<mg::DynFn, mg::DynFn, mg::DynProp, 8>(a); }\n'
           'extern "C" __global__ void k_rj(const __grid_constant__ mg::RjArgs a) { mg::rj_ensemble_body<8>(a); }\n'
           'extern "C" __global__ void k_ni(mg::NestArgs a, double *x, double *ll, double *lp) { mg::nest_init_body<8>(a, x, ll, lp); }\n'
           'extern "C" __global__ void k_nr(mg::NestArgs a, mg::NestProp p, int s0, int s1, int f, int l, double *cx, double *cl) { mg::nest_replace_simple_body<8>(a, p, s0, s1, f, l, cx, cl); }\n')
    prog = ctypes.c_void_p()
    hn = (ctypes.c_char_p * len(names))(*[n.encode() for n in names])
    hs = (ctypes.c_char_p * len(names))(*[s.encode() for s in srcs])
    assert nv.nvrtcCreateProgram(ctypes.byref(prog), src.encode(), b"t.cu", len(names), hs, hn) == 0
    opts = [b"--gpu-architecture=sm_100a", b"--std=c++17", b"--fmad=false", b"-default-device"]
    rc = nv.nvrtcCompileProgram(prog, len(opts), (ctypes.c_char_p * len(opts))(*opts))
    n = ctypes.c_size_t()
    nv.nvrtcGetProgramLogSize(prog, ctypes.byref(n))
    log = ctypes.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(prog, log)
    assert rc == 0, log.value.decode()[:2000]


def test_ocaml_externals_have_the_arity_of_their_stubs():
    """Without an OCaml compiler the one mistake a reader is likely to miss is an `external` whose number of arguments
    differs from its C stub's: count the arrows of every external's type (outside parentheses) against the `value`
    parameters of the native stub; externals with more than five arguments must name a bytecode stub first."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    c_text = open(os.path.join(root, "ocaml", "mcmc_gpu_stubs.c")).read()
    ml = open(os.path.join(root, "ocaml", "mcmc_gpu.ml")).read()
    prims = {m.group(1): len(re.findall(r"\bvalue\s+\w+", m.group(2)))
             for m in re.finditer(r"CAMLprim\s+value\s+(\w+)\s*\(([^)]*)\)", c_text)}
    checked = 0
    for m in re.finditer(r"external\s+(\w+)\s*:\s*(.*?)=\s*((?:\"\w+\"\s*)+)", ml, re.S):
        name, typ, stubs = m.group(1), m.group(2), re.findall(r'"(\w+)"', m.group(3))
        depth, arrows, i = 0, 0, 0
        while i < len(typ):                       # arrows at nesting depth 0 = arguments
            ch = typ[i]
            if ch in "([":
                depth += 1
            elif ch in ")]":
                depth -= 1
            elif typ.startswith("->", i) and depth == 0:
                arrows += 1
                i += 1
            i += 1
        native = stubs[-1]
        assert native in prims, (name, native)
        assert prims[native] == arrows, f"external {name}: {arrows} arguments, stub {native} takes {prims[native]}"
        if arrows > 5:
            assert len(stubs) == 2 and stubs[0].endswith("_bytecode"), f"external {name} needs a bytecode stub"
            assert prims[stubs[0]] == 1 or "value *" in c_text[c_text.index(stubs[0]):c_text.index(stubs[0]) + 80], stubs[0]
        else:
            assert len(stubs) == 1, f"external {name}: {arrows} arguments need no bytecode stub"
        checked += 1
    assert checked >= 20


def test_environment_switches_match_design_table():
    """the MCMC_GPU_* variables the package reads are exactly those DESIGN.md section 7a lists"""
    import os
    import re
    pkg = os.path.dirname(os.path.abspath(_abi.__file__))
    root = os.path.dirname(pkg)
    read = set()
    for d, dirs, files in os.walk(pkg):
        dirs[:] = [x for x in dirs if x not in ("build", "__pycache__")]
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h")):
                text = open(os.path.join(d, f), encoding="utf-8").read()
                read |= set(re.findall(r'(?:getenv|os\.environ(?:\.get)?)\s*[(\[]\s*"(MCMC_GPU_\w+)"', text))
    design = open(os.path.join(root, "DESIGN.md"), encoding="utf-8").read()
    section = design[design.index("\n## 7a."):]
    section = section[:section.index("\n## ", 1)]
    listed = {m for line in section.splitlines() if line.startswith("|") for m in re.findall(r"MCMC_GPU_\w+", line)}
    assert read == listed, f"read but not listed: {sorted(read - listed)}; listed but not read: {sorted(listed - read)}"
