"""CPU: the code generator of the specialised forward kernel (neurodiffeq_b200/jit.py).  The generated straight-line source of
every traced program of the BASELINE and extension workloads is compiled FOR THE HOST (device intrinsics replaced by their
host meaning) and run on random inputs; it must agree with a numpy restatement of the bytecode interpreter
(csrc/pinnjet_program.cuh) -- operation by operation the same float32 arithmetic, so the comparison is tight."""
import os
import subprocess
import zlib

import numpy as np
import pytest

import workloads
from helpers import product_namespace

HARNESS = r'''
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#define __device__
#define __forceinline__ inline
static inline float __int_as_float(int v) { float f; std::memcpy(&f, &v, 4); return f; }
static inline float __ldg(const float* p) { return *p; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
struct ProgIO {
    const float* const* coords; long long gidx; long long N; const float* ycache; int ystride; const float* rbar; float loss_scale;
    float* u_out; float* r_out; float* seed_tile; int T; float* w_out = nullptr; int w_stride = 0; int slot_stride = 0;
};
namespace pj {
#include "prog.inc"
}
int main(int argc, char** argv) {
    // stdin: n_coords N n_y loss_scale, then coords [n_coords][N], ycache [n_y]; stdout: u[8] r[8] seed[32] w[16] sumsq
    int nc, N, ny; float ls;
    if (scanf("%d %d %d %f", &nc, &N, &ny, &ls) != 4) return 1;
    float* c = (float*)calloc((size_t)nc * N, 4); float* y = (float*)calloc(ny + 1, 4);
    for (int i = 0; i < nc * N; ++i) if (scanf("%f", c + i) != 1) return 1;
    for (int i = 0; i < ny; ++i) if (scanf("%f", y + i) != 1) return 1;
    const float* cp[16]; for (int i = 0; i < nc; ++i) cp[i] = c + (size_t)i * N;
    float u[8 * 4] = {0}, r[8 * 4] = {0}, seed[64] = {0}, w[32] = {0};
    ProgIO io{cp, 1, N, y, 1, nullptr, ls, u, r, seed, 1};
    io.N = 1; io.gidx = 0;                       // outputs are [row][N]: one point, so row strides are 1
    const float* cp1[16]; for (int i = 0; i < nc; ++i) cp1[i] = c + (size_t)i * N + 1; io.coords = cp1;
    io.w_out = w; io.w_stride = 1;
    float s = pj::PROG(io);
    for (int i = 0; i < 8; ++i) printf("%.9g ", u[i]);
    for (int i = 0; i < 8; ++i) printf("%.9g ", r[i]);
    for (int i = 0; i < 32; ++i) printf("%.9g ", seed[i]);
    for (int i = 0; i < 16; ++i) printf("%.9g ", w[i]);
    printf("%.9g\n", s);
    return 0;
}
'''


@pytest.mark.parametrize("key", ["c1", "c2", "c3", "c4", "c5", "x1", "x5", "x7"])
def test_generated_programs_match_the_interpreter(key, tmp_path):
    from neurodiffeq_b200 import jit
    from neurodiffeq_b200.engine import combine_seconds
    from neurodiffeq_b200.tracing import TracedProblem
    wl = workloads.build(product_namespace(), key)
    tp = TracedProblem(wl.make_nets(), wl.make_conditions(), workloads.bundle_eq_wrapper(wl), len(wl.coord_names),
                       combine_seconds=combine_seconds)
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    n_coords, n_pts = tp.n_coords, 3
    for name, prog in (("train", tp.prog_train), ("eval", tp.prog_eval), ("w", tp.prog_w if tp.wl else None)):
        if prog is None:
            continue
        src = jit.program_source("PROG_FN", prog)
        (tmp_path / "prog.inc").write_text(src)
        (tmp_path / "h.cpp").write_text(HARNESS.replace("pj::PROG(io)", "pj::PROG_FN(io)"))
        exe = tmp_path / f"h_{name}"
        subprocess.check_call(["g++", "-O0", "-ffp-contract=off", "-I", str(tmp_path), str(tmp_path / "h.cpp"), "-o", str(exe)])
        n_y = int(max([z for op, y, z, w in prog.code.tolist() if op == 2], default=0)) + 1
        coords = rng.uniform(0.2, 1.3, size=(n_coords, n_pts)).astype(np.float32)
        ycache = rng.normal(size=n_y).astype(np.float32)
        text = f"{n_coords} {n_pts} {n_y} 0.37\n" + " ".join(repr(float(v)) for v in coords.reshape(-1)) + "\n" + \
               " ".join(repr(float(v)) for v in ycache) + "\n"
        out = np.array(subprocess.check_output([str(exe)], input=text.encode()).split(), dtype=np.float64)
        ref = jit.numpy_reference(prog, coords, 1, ycache, loss_scale=np.float32(0.37))
        got = {"u": out[0:8], "r": out[8:16], "seed": out[16:48], "w": out[48:64]}
        for kind in ("u", "r", "seed", "w"):
            for row, val in ref[kind].items():
                assert got[kind][row] == pytest.approx(val, rel=1e-4, abs=1e-5), (key, name, kind, row)   # libm vs numpy ulps, amplified by cancellation
        assert out[64] == pytest.approx(sum(v * v for v in ref["r"].values()), rel=1e-3, abs=1e-8)


def test_module_source_names_the_scheme_and_refuses_trainable_immediates():
    from neurodiffeq_b200 import jit
    from neurodiffeq_b200.engine import combine_seconds
    from neurodiffeq_b200.tracing import TracedProblem
    wl = workloads.build(product_namespace(), "c2")
    tp = TracedProblem(wl.make_nets(), wl.make_conditions(), workloads.bundle_eq_wrapper(wl), 2, combine_seconds=combine_seconds)
    head, body = jit.module_source(tp)
    assert "#define PJ_JIT_N1 2" in head and "#define PJ_JIT_N2 1" in head and "#define PJ_JIT_WL 2" in head
    assert "pj_jit_program_train" in body and "pj_jit_program_eval" in body and "pj_jit_program_w" in body
    wl9 = workloads.build(product_namespace(), "x9")                       # Resnet: shortcut weights are program immediates
    tp9 = TracedProblem(wl9.make_nets(), wl9.make_conditions(), workloads.bundle_eq_wrapper(wl9), len(wl9.coord_names),
                        combine_seconds=combine_seconds)
    with pytest.raises(ValueError, match="trainable immediates"):
        jit.module_source(tp9)


@pytest.mark.skipif(not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="no nvcc")
def test_specialised_kernel_compiles_for_sm_100a(tmp_path, monkeypatch):
    from neurodiffeq_b200 import jit
    from neurodiffeq_b200.engine import combine_seconds
    from neurodiffeq_b200.tracing import TracedProblem
    monkeypatch.setattr(jit, "CACHE", str(tmp_path))
    wl = workloads.build(product_namespace(), "c5")
    tp = TracedProblem(wl.make_nets(), wl.make_conditions(), workloads.bundle_eq_wrapper(wl), len(wl.coord_names),
                       combine_seconds=combine_seconds)
    data, key = jit.compile_cubin(tp)
    assert data[:4] == b"\x7fELF" and os.path.exists(os.path.join(str(tmp_path), key + ".cubin"))
    data2, key2 = jit.compile_cubin(tp)                                    # second call: served from the cache
    assert key2 == key and data2 == data
    monkeypatch.setattr(jit, "_cache_dir", lambda: None)                   # no trustworthy cache directory: compile, keep nothing
    os.remove(os.path.join(str(tmp_path), key + ".cubin"))
    data3, key3 = jit.compile_cubin(tp)
    assert key3 == key and data3[:4] == b"\x7fELF" and os.listdir(str(tmp_path)) == []


def test_cache_falls_back_to_a_private_temporary_directory(tmp_path, monkeypatch):
    """A cache directory that cannot be created (no writable home) moves the cubin cache to a per-user directory under the
    temporary directory, created private.  A cached cubin runs in the caller's CUDA context, so a directory another account
    could write to -- world-writable, owned by someone else, or a symlink -- is never used: no caching then."""
    import tempfile
    from neurodiffeq_b200 import jit
    blocker = tmp_path / "not_a_directory"
    blocker.write_text("")
    monkeypatch.setattr(jit, "CACHE", str(blocker / "pinnjet_jit"))
    tmp = tmp_path / "tmp"
    os.makedirs(str(tmp))
    monkeypatch.setattr(tempfile, "tempdir", str(tmp))
    fallback = os.path.join(str(tmp), f"pinnjet_jit-{os.getuid()}")
    assert jit._cache_dir() == fallback and os.stat(fallback).st_mode & 0o077 == 0

    os.chmod(fallback, 0o777)                                              # planted world-writable
    assert jit._cache_dir() is None
    os.rmdir(fallback)
    os.makedirs(str(tmp_path / "elsewhere"), mode=0o700)
    os.symlink(str(tmp_path / "elsewhere"), fallback)                     # planted symlink
    assert jit._cache_dir() is None
    os.remove(fallback)
    real_uid = os.getuid()
    monkeypatch.setattr(os, "getuid", lambda: real_uid + 1)               # a private directory of ANOTHER account
    os.makedirs(os.path.join(str(tmp), f"pinnjet_jit-{real_uid + 1}"), mode=0o700)
    assert jit._cache_dir() is None
    monkeypatch.setattr(os, "getuid", lambda: real_uid)

    monkeypatch.setattr(jit, "CACHE", str(tmp_path / "home_cache"))       # a usable CACHE comes first
    assert jit._cache_dir() == str(tmp_path / "home_cache")
