"""CPU test: the ggml hook replacement (t-mac_b200/ggml/ggml-tmac.cpp) compiles against the REFERENCE's own ggml.h /
ggml-tmac.h and, together with libtmac_b200.so, resolves all ten hook symbols with the reference prototypes
(3rdparty/llama.cpp/ggml/include/ggml-tmac.h:25-38).  The same checks run against the restatement of those declarations in
tests/ggml_headers (every checkout) and against the upstream headers where that tree is present; no compute call is made (no GPU
needed)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_INC = "/root/reference/3rdparty/llama.cpp/ggml/include"
STORED_INC = os.path.join(ROOT, "tests", "ggml_headers")
LIB_DIR = os.path.join(ROOT, "t-mac_b200")

MAIN = r'''
#include "ggml-tmac.h"
#define TMAC_B200_NO_GGML_DECLS
#include "tmac_b200.h"
#include <stdio.h>
int main(void) {
    tmac_b200_kcfg k = {11008, 4096, 2, 128, 16, 16, 8, 128, 64, 1, 0};   /* what kcfg.ini provides in the reference */
    if (tmac_b200_register_kcfg(&k) != 0) return 2;
    /* every hook of ggml-tmac.h:25-38, taken by address through the reference prototypes */
    void *syms[] = {(void *)ggml_tmac_init, (void *)ggml_tmac_free, (void *)ggml_tmac_can_mul_mat, (void *)ggml_tmac_mul_mat_get_wsize,
                    (void *)ggml_tmac_mul_mat_task_init, (void *)ggml_tmac_mul_mat_task_compute, (void *)ggml_tmac_transform_tensor,
                    (void *)ggml_tmac_get_type_bits, (void *)ggml_tmac_set_n_threads, (void *)ggml_tmac_get_nbytes};
    int n = 0;
    for (unsigned i = 0; i < sizeof syms / sizeof syms[0]; ++i) n += syms[i] != 0;
    /* host-only calls (no CUDA): type bits, workspace size and nbytes arithmetic as in ggml-tmac.cpp:250-288,503-526 */
    struct ggml_tensor w = {0}, x = {0};
    w.type = GGML_TYPE_I2; w.ne[0] = 4096; w.ne[1] = 11008; x.type = GGML_TYPE_F32; x.ne[0] = 4096; x.ne[1] = 1;
    printf("%d %d %zu %zu\n", n, ggml_tmac_get_type_bits(GGML_TYPE_I2), ggml_tmac_mul_mat_get_wsize(&w, &x, &x), ggml_tmac_get_nbytes(&w));
    return 0;
}
'''


def _shim_compiles_and_resolves_all_hooks(tmp_path, inc):
    assert os.path.exists(os.path.join(LIB_DIR, "libtmac_b200.so")), "build the library first"
    obj = tmp_path / "ggml-tmac.o"
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-Wall", "-Werror", "-c", os.path.join(LIB_DIR, "ggml", "ggml-tmac.cpp"),
                    "-I", inc, "-I", os.path.join(ROOT, "include"), "-o", str(obj)], check=True)
    main_c = tmp_path / "main.c"
    main_c.write_text(MAIN)
    main_o = tmp_path / "main.o"
    subprocess.run(["gcc", "-O1", "-c", str(main_c), "-I", inc, "-I", os.path.join(ROOT, "include"), "-o", str(main_o)], check=True)
    exe = tmp_path / "hooks"
    subprocess.run(["g++", str(main_o), str(obj), "-L", LIB_DIR, "-ltmac_b200", "-Wl,-rpath," + LIB_DIR, "-Wl,--no-undefined", "-o", str(exe)], check=True)
    # the four tensor-taking hooks come from the shim, the other six from the shared library
    nm = subprocess.run(["nm", "-D", "--defined-only", os.path.join(LIB_DIR, "libtmac_b200.so")], check=True, capture_output=True, text=True).stdout
    for s in ("ggml_tmac_init", "ggml_tmac_free", "ggml_tmac_mul_mat_task_init", "ggml_tmac_mul_mat_task_compute", "ggml_tmac_set_n_threads", "ggml_tmac_get_type_bits"):
        assert (" T " + s + "\n") in nm, s
    nmo = subprocess.run(["nm", "--defined-only", str(obj)], check=True, capture_output=True, text=True).stdout
    for s in ("ggml_tmac_can_mul_mat", "ggml_tmac_mul_mat_get_wsize", "ggml_tmac_transform_tensor", "ggml_tmac_get_nbytes"):
        assert (" T " + s + "\n") in nmo, s
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert out[0] == "10" and out[1] == "2"
    # wsize / nbytes: the reference's formulas (ggml-tmac.cpp:258-263: qlut K*N*4 + 2 * lut scales/biases; :277-288: M*K*bits/8 + scales)
    assert int(out[2]) == 4096 * 4 + 2 * 64 * 4 and int(out[3]) == 11008 * 4096 * 2 // 8 + 11008 * 32 * 2 * 4


@pytest.mark.skipif(not os.path.isdir(REF_INC), reason="reference headers not mounted (GPU box)")
def test_shim_compiles_against_reference_headers_and_resolves_all_hooks(tmp_path):
    _shim_compiles_and_resolves_all_hooks(tmp_path, REF_INC)


def test_shim_compiles_against_stored_hook_declarations_and_resolves_all_hooks(tmp_path):
    _shim_compiles_and_resolves_all_hooks(tmp_path, STORED_INC)


@pytest.mark.skipif(not os.path.isdir(REF_INC), reason="reference tree not mounted (GPU box)")
def test_vendored_ggml_builds_with_GGML_TMAC_against_this_package(tmp_path):
    """SURVEY 8 f4: the reference's vendored ggml configured with -DGGML_TMAC=ON -DGGML_TMAC_TVM_THREADPOOL=ON (the branch of
    ggml.c that calls the hook once per mat-vec from thread 0, ref:ggml.c:12610-12630) finds package TMAC = this library,
    compiles our ggml-tmac.cpp in place of the reference's and links libtmac_b200.so (tools/ggml_tmac_build.sh)."""
    env = dict(os.environ, W=str(tmp_path / "w"))
    r = subprocess.run(["bash", os.path.join(ROOT, "tools", "ggml_tmac_build.sh")], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "TMAC found" in r.stdout and "ggml_tmac_* symbols defined in libggml: 4" in r.stdout
    for s in ("ggml_tmac_init", "ggml_tmac_mul_mat_task_init", "ggml_tmac_mul_mat_task_compute", "ggml_tmac_get_type_bits"):
        assert s in r.stdout, s                  # imported by libggml.so, exported by libtmac_b200.so
    assert "libtmac_b200.so" in r.stdout
