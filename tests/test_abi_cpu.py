"""The C-ABI shared library builds for sm_100a, loads, exports every symbol include/lirec_b200.h
declares, and refuses to compute without a B200 (no CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lirec_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(built_lib):
    lib = ctypes.CDLL(built_lib)
    declared = _declared_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), "include/lirec_b200.h declares %s but the library does not export it" % name


def test_binding_lists_every_symbol_of_abi_version_3(built_lib):
    """Version 3: lirec_rows_expand_bwd reads the ReLU gate as the bit mask of LIREC_POST_SIGN_MASK and writes
    only the transposed hi/lo form, and lirec_split_f32 writes the transposed split.  The symbol list is that
    of version 2."""
    from lirec_b200 import _ext
    assert sorted(_ext.EXPORTED_SYMBOLS) == _declared_symbols()
    assert _ext.lib().lirec_abi_version() == 3


def test_sass_is_blackwell_native(built_lib):
    """tcgen05.mma / TMA / TMEM loads show up as UTCHMMA / UTMALDG / LDTM in the SASS."""
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "HMMA." not in sass.replace("UTCHMMA", ""), "legacy mma.sync path found"


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu(built_lib):
    from lirec_b200 import _ext, ops
    with pytest.raises(RuntimeError, match="no CPU"):
        _ext.require_device()
    x = torch.zeros(4, 8)
    with pytest.raises(RuntimeError):
        ops.cast_bf16(x, torch.zeros(4, 8, dtype=torch.bfloat16))
    # the raw entry points refuse too
    rc = _ext.lib().lirec_cast_bf16(None, None, 0, None)
    assert rc != 0 and b"CPU fallback" in _ext.lib().lirec_last_error() or rc != 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_model_refuses_cpu(built_lib, opt_preset):
    opt_preset("int_rel_ch", device="cpu")
    import lirec_b200.mlp.model as M
    with pytest.raises(RuntimeError, match="no CPU"):
        M.create_model(101, n_rels=15)


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under lirec_b200/ may import it."""
    pkg = os.path.join(ROOT, "lirec_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith(".py"):
                with open(os.path.join(dirpath, fn)) as f:
                    src = f.read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, fn)


def test_integration_stubs_match_the_binding():
    """INTEGRATION.md's ctypes stubs: every python block parses, and the struct it declares has the fields of
    the real binding (a by-value struct with missing tail fields would pass garbage)."""
    from lirec_b200 import _ext
    with open(os.path.join(ROOT, "INTEGRATION.md")) as f:
        blocks = re.findall(r"```python\n(.*?)```", f.read(), flags=re.S)
    assert len(blocks) >= 3
    for b in blocks:
        compile(b, "INTEGRATION.md", "exec")
    stub = [b for b in blocks if "class TrackLossCfg" in b][0]
    fields = re.findall(r'\("(\w+)", ctypes\.c_(\w+)\)', stub.split("def margin_track_rels")[0])
    real = list(_ext.TrackLossCfg._fields_)
    assert [(n, getattr(ctypes, "c_" + t)) for n, t in fields] == real, (fields, real)
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        header = f.read()
    body = header[header.index("typedef struct lirec_track_loss_cfg"):header.index("} lirec_track_loss_cfg;")]
    assert re.findall(r"\b(?:float|int32_t|uint32_t)\s+(\w+);", body) == [n for n, _ in real]


def test_header_is_plain_c_and_struct_layouts_match_ctypes(tmp_path):
    """include/lirec_b200.h compiles as C (gcc, no CUDA headers), and every struct the ctypes binding passes
    has the size and the field offsets the C compiler gives it."""
    import shutil
    import subprocess
    from lirec_b200 import _ext
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    pairs = {"lirec_dropout": _ext.Dropout, "lirec_operand": _ext.Operand, "lirec_gemm_pass": _ext.GemmPass,
             "lirec_epilogue": _ext.Epilogue, "lirec_gemm_problem": _ext.GemmProblem,
             "lirec_track_loss_cfg": _ext.TrackLossCfg, "lirec_linear": _ext.Linear, "lirec_encoder": _ext.Encoder,
             "lirec_model_params": _ext.ModelParams, "lirec_model_cfg": _ext.ModelCfg, "lirec_batch": _ext.Batch}
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        header = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lirec_b200.h"', "int main(void) {"]
    expect = []
    for cname, ct in pairs.items():
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), header, flags=re.S).group(1)
        # `a, b` declarations: the first name is the last token of the part before the first comma
        cfields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            parts = [x.strip() for x in decl.split(",")]
            names = [parts[0].split()[-1]] + parts[1:]
            cfields += [re.sub(r"\[.*", "", n).lstrip("*") for n in names]
        pfields = [n for n, _ in ct._fields_]
        assert len(cfields) == len(pfields), (cname, cfields, pfields)
        lines.append('printf("%%zu\\n", sizeof(%s));' % cname)
        expect.append((cname, "sizeof", ctypes.sizeof(ct)))
        for cf, pf in zip(cfields, pfields):
            lines.append('printf("%%zu\\n", offsetof(%s, %s));' % (cname, cf))
            expect.append((cname, cf, getattr(ct, pf).offset))
    lines += ["return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert len(out) == len(expect)
    for got, (cname, what, want) in zip(out, expect):
        assert int(got) == want, (cname, what, got, want)


def test_argtypes_arity_matches_the_header(built_lib):
    """Every entry point the binding types has as many `argtypes` as the header declares parameters, with
    pointers / 64-bit / 32-bit / float / by-value-struct parameters in the same positions."""
    from lirec_b200 import _ext
    L = _ext.lib()
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        header = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    decls = re.findall(r"\b(lirec_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", header)
    assert len(decls) >= 25
    checked = 0
    for name, params in decls:
        params = [p.strip() for p in params.split(",")] if params.strip() not in ("", "void") else []
        fn = getattr(L, name)
        if fn.argtypes is None:
            assert not params or name == "lirec_profile_begin", name
            continue
        assert len(fn.argtypes) == len(params), (name, len(fn.argtypes), params)
        for at, p in zip(fn.argtypes, params):
            if "*" in p:
                kind = ctypes.c_void_p
            elif re.match(r"(const\s+)?(int64_t|size_t)\b", p):
                kind = (ctypes.c_int64, ctypes.c_size_t)
            elif re.match(r"(const\s+)?(int32_t|int|uint32_t)\b", p):
                kind = (ctypes.c_int32, ctypes.c_uint32, ctypes.c_int)
            elif re.match(r"(const\s+)?float\b", p):
                kind = ctypes.c_float
            else:                                   # a struct by value
                assert issubclass(at, ctypes.Structure), (name, p, at)
                continue
            assert at in (kind if isinstance(kind, tuple) else (kind,)), (name, p, at)
        checked += 1
    assert checked >= 20
