"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol the headers
declare, the reference's unmodified driver compiles against include/ray.h, and the product path fails
loudly (no fallback) when there is no GPU."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_MAIN_BIN = os.path.join(ROOT, "oracle", "_ref", "main_ref")


def header_functions(path):
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:futhark|ray_b200)_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol(R):
    lib = ctypes.CDLL(R.lib_path())
    declared = header_functions(os.path.join(ROOT, "include", "ray.h")) + header_functions(os.path.join(ROOT, "include", "ray_b200.h"))
    assert len(declared) > 50
    missing = [f for f in declared if not hasattr(lib, f)]
    assert not missing, f"declared in include/*.h but not exported: {missing}"


def test_reference_driver_symbols_are_exported(R):
    # the 14 functions futhark/main.c calls (main.c:59-141; SURVEY.md §8b)
    need = ["futhark_context_config_new", "futhark_context_config_free", "futhark_context_new", "futhark_context_free",
            "futhark_context_get_error", "futhark_context_sync", "futhark_entry_rgbbox", "futhark_entry_irreg",
            "futhark_entry_prepare_scene", "futhark_entry_render", "futhark_values_i32_2d", "futhark_free_i32_2d",
            "futhark_free_opaque_prepared_scene", "futhark_free_opaque_scene"]
    lib = ctypes.CDLL(R.lib_path())
    assert all(hasattr(lib, f) for f in need)


def test_python_binding_covers_the_headers(R):
    declared = set(header_functions(os.path.join(ROOT, "include", "ray.h")) + header_functions(os.path.join(ROOT, "include", "ray_b200.h")))
    bound = set(R.declared_symbols())
    # everything bound must be declared; config-only helpers may stay unbound
    assert bound <= declared, bound - declared


def test_struct_layouts_match_the_library(R):
    """ctypes mirrors of the C structs have the size the library was compiled with (no GPU needed)."""
    lib = R.load_library()
    assert ctypes.sizeof(R.RenderJob) == lib.ray_b200_render_job_size() == 72


def test_tuning_parameters_match_the_documented_environment_variables(R):
    """futhark_get_tuning_param_* / futhark_context_config_set_tuning_param (host-only calls): every RAY_* variable of
    INTEGRATION.md's tuning rows exists as a tuning parameter of the same name, unknown names are rejected."""
    lib = R.load_library()
    lib.futhark_get_tuning_param_name.restype = ctypes.c_char_p
    names = {lib.futhark_get_tuning_param_name(i).decode() for i in range(lib.futhark_get_tuning_param_count())}
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    rows = [ln for ln in text.splitlines() if ln.startswith("| `RAY_") and "tuning" in ln]
    documented = {v.lower() for ln in rows for v in re.findall(r"`RAY_(\w+)`", ln.split("|")[1])}
    assert {"wq_low", "wq_ncap", "wq_packet", "stage_cap", "lw_slots"} <= documented
    assert documented <= names, documented - names
    lib.futhark_context_config_new.restype = ctypes.c_void_p
    cfg = ctypes.c_void_p(lib.futhark_context_config_new())
    try:
        for n in sorted(names):
            assert lib.futhark_context_config_set_tuning_param(cfg, n.encode(), ctypes.c_size_t(1)) == 0, n
        assert lib.futhark_context_config_set_tuning_param(cfg, b"no_such_parameter", ctypes.c_size_t(1)) != 0
    finally:
        lib.futhark_context_config_free(cfg)


def _compile(src, out, extra=()):
    cmd = ["/usr/bin/gcc", "-O3", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", src, "-o", out,
           "-I" + os.path.join(ROOT, "include"), "-L" + os.path.join(ROOT, "raytracers_b200"), "-lray_b200",
           "-Wl,-rpath," + os.path.join(ROOT, "raytracers_b200"), "-lm", *extra]
    return subprocess.run(cmd, capture_output=True, text=True)


@pytest.mark.skipif(not os.path.exists(REF_MAIN_BIN), reason="oracle/_ref/main_ref not built (no checkout of the original project)")
def test_unmodified_reference_main_c_compiles_and_links(R):
    # build() compiles it with the same flags as futhark/Makefile:13-14,21 plus -Werror (oracle/Makefile, `make ref`);
    # here: the binary it made resolves this repository's library
    out = subprocess.run(["ldd", REF_MAIN_BIN], capture_output=True, text=True).stdout
    linked = [ln.split("=>")[1].split()[0] for ln in out.splitlines() if ln.strip().startswith("libray_b200.so =>")]
    want = os.path.realpath(os.path.join(ROOT, "raytracers_b200", "libray_b200.so"))
    assert [os.path.realpath(p) for p in linked] == [want], out


def test_repo_driver_compiles_and_links(tmp_path, R):
    r = _compile(os.path.join(ROOT, "examples", "driver.c"), str(tmp_path / "driver"))
    assert r.returncode == 0, r.stderr


def _no_gpu():
    try:
        import torch
        return not torch.cuda.is_available()
    except Exception:
        return True


@pytest.mark.skipif(not _no_gpu(), reason="only meaningful on a machine without a GPU")
def test_no_cpu_fallback(R, tmp_path):
    with pytest.raises(R.RayError, match="no CPU fallback"):
        R.Context()
    # the C driver must fail too (main.c:64 asserts get_error == NULL)
    r = _compile(os.path.join(ROOT, "examples", "driver.c"), str(tmp_path / "driver"))
    assert r.returncode == 0
    run = subprocess.run([str(tmp_path / "driver"), "-n", "8", "-m", "8", "-r", "1"], capture_output=True, text=True)
    assert run.returncode != 0 and "no CPU fallback" in run.stderr


def test_product_never_touches_the_oracle():
    import ast
    pkg = os.path.join(ROOT, "raytracers_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py"):
                for node in ast.walk(ast.parse(open(path).read())):
                    names = []
                    if isinstance(node, ast.Import):
                        names = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        names = [node.module or ""]
                    assert not any("oracle" in n for n in names), (path, names)
            elif f.endswith((".cu", ".cuh", ".cpp", ".h")) or f == "Makefile":
                for line in open(path, errors="replace"):
                    if line.lstrip().startswith("#include") or "dlopen" in line or "liboracle" in line:
                        assert "oracle" not in line, (path, line)
    out = subprocess.run(["ldd", os.path.join(pkg, "libray_b200.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out
