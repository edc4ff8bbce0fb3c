"""The C-ABI library builds for sm_100a, loads, and exports every symbol include/afs_b200.h declares."""
import ctypes
import os
import re
import subprocess

from conftest import ROOT


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "afs_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(afs_[a-z0-9_]+)\s*\(", text)))


def test_build_and_exports():
    from audio_fewshot_b200 import build
    path = build.build()
    assert os.path.exists(path)
    handle = ctypes.CDLL(path)
    names = declared_symbols()
    assert len(names) >= 15
    for name in names:
        assert hasattr(handle, name), "missing export %s" % name
    handle.afs_abi_version.restype = ctypes.c_int
    assert handle.afs_abi_version() == 1
    handle.afs_status_string.restype = ctypes.c_char_p
    assert handle.afs_status_string(-4) == b"workspace too small"


def test_binding_covers_header():
    from audio_fewshot_b200 import _lib
    assert sorted(_lib.SIGNATURES.keys()) == declared_symbols()
    h = _lib.lib()  # loads and type-checks every symbol
    assert h.afs_proto_workspace_bytes(1, 5, 5, 1600) == 5 * 1600 * 4 + 32  # prototypes + 5 inverse norms, 16-byte padded
    assert h.afs_proto_workspace_bytes(2, 5, 1, 12800) == 2 * 5 * 12800 * 4 + 48
    assert h.afs_dn4_workspace_bytes(100, 1, 5, 5, 64, 20) > 100 * 64 * 20 * 4


def test_sass_is_sm100a():
    from audio_fewshot_b200 import build
    path = build.build()
    out = subprocess.run(["cuobjdump", "-lelf", path], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_invalid_arguments_are_rejected_without_a_gpu():
    from audio_fewshot_b200 import _lib
    h = _lib.lib()
    # null pointers / bad sizes must be refused before any CUDA call
    assert h.afs_proto_fwd(None, 0, None, 0, 0, 5, 5, 1600, 0, None, None, None, 0, None) == -1
    assert h.afs_vote_acc(None, 5, None, 0, None, 1, None, None, None, None) == -1
    assert h.afs_bdc_fwd(None, 1, 64, 10, None, 1, None, None) == -1


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "audio_fewshot_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f
                assert "/root/reference" not in src, f


def test_header_is_plain_c_and_a_c_host_links(tmp_path):
    """include/afs_b200.h must be usable from a C host (no C++ or torch types in any signature): a C99 translation
    unit that includes it, takes the address of every declared entry point and calls the GPU-free ones compiles with
    gcc, links against libafs_b200.so and runs."""
    from audio_fewshot_b200 import build
    lib = build.build()
    names = declared_symbols()
    src = tmp_path / "host.c"
    src.write_text(
        '#include <stdio.h>\n#include "afs_b200.h"\n'
        "typedef void (*fn_t)(void);\n"
        "int main(void) {\n"
        "  fn_t fns[] = {%s};\n"
        "  size_t n = sizeof(fns) / sizeof(fns[0]);\n"
        "  for (size_t i = 0; i < n; ++i) if (fns[i] == 0) return 2;\n"
        "  if (afs_abi_version() != AFS_ABI_VERSION) return 3;\n"
        "  if (afs_proto_fwd(0, 0, 0, 0, 0, 5, 5, 1600, 0, 0, 0, 0, 0, 0) != AFS_ERR_INVALID_ARG) return 4;\n"
        '  printf("%%s %%zu\\n", afs_status_string(AFS_ERR_WORKSPACE), n);\n'
        "  return 0;\n}\n" % ", ".join("(fn_t)%s" % n for n in names))
    exe = tmp_path / "host"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), lib, "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out
    assert out.stdout.split() == ["workspace", "too", "small", str(len(names))]


def test_conv3x3_weight_packing_layout_and_tf32_rounding():
    """afs_conv3x3_c64_pack_weights is host code: check on the CPU that the operand layout holds the weights where
    the kernel expects them -- [tap][kc][chunk][cout][4] -- and that values are rounded to the nearest TF32 (ties away
    from zero, what cvt.rna.tf32 does)."""
    import numpy as np
    from audio_fewshot_b200 import _lib
    h = _lib.lib()
    rng = np.random.default_rng(0)
    w = (rng.standard_normal((64, 64, 3, 3)) * 0.1).astype(np.float32)
    w[0, 0, 0, 0] = np.float32(1.0) + np.float32(2.0 ** -11)  # exactly half a TF32 ulp above 1: rounds away from zero
    n = int(h.afs_conv3x3_c64_packed_floats())
    assert n == 9 * 8 * 2 * 64 * 4
    packed = np.empty(n, np.float32)
    assert h.afs_conv3x3_c64_pack_weights(w.ctypes.data_as(ctypes.c_void_p), packed.ctypes.data_as(ctypes.c_void_p)) == 0
    bits = w.view(np.uint32).astype(np.uint64)
    want = (((bits + 0x1000) & ~np.uint64(0x1FFF)).astype(np.uint32)).view(np.float32)  # [co][ci][ky][kx]
    assert want[0, 0, 0, 0] == np.float32(1.0) + np.float32(2.0 ** -10)
    ref = want.reshape(64, 8, 2, 4, 9)                      # [co][kc][chunk][i][tap]  (ci = 8 kc + 4 chunk + i)
    assert np.array_equal(packed.reshape(9, 8, 2, 64, 4), ref.transpose(4, 1, 2, 0, 3))  # [tap][kc][chunk][cout][i]
    assert h.afs_conv3x3_c64_pack_weights(None, packed.ctypes.data_as(ctypes.c_void_p)) == -1


def test_conv3x3_bf16_weight_packing_layout_and_rounding():
    """afs_conv3x3_c64_pack_weights_bf16 (host code): [tap][kc][chunk][cout][8] with cin = 16 kc + 8 chunk + i, values
    rounded to the nearest bf16, ties to even -- torch's float32 -> bfloat16 conversion."""
    import numpy as np
    import torch
    from audio_fewshot_b200 import _lib
    h = _lib.lib()
    rng = np.random.default_rng(1)
    w = (rng.standard_normal((64, 64, 3, 3)) * 0.1).astype(np.float32)
    w[0, 0, 0, 0] = np.float32(1.0) + np.float32(2.0 ** -8)   # a tie: rounds to the even neighbour 1.0
    w[0, 1, 0, 0] = np.float32(1.0) + np.float32(3 * 2.0 ** -8)  # a tie: rounds up to 1 + 2^-6
    n = int(h.afs_conv3x3_c64_packed_bf16_elems())
    assert n == 9 * 4 * 2 * 64 * 8
    packed = np.empty(n, np.uint16)
    assert h.afs_conv3x3_c64_pack_weights_bf16(w.ctypes.data_as(ctypes.c_void_p), packed.ctypes.data_as(ctypes.c_void_p)) == 0
    want = torch.from_numpy(w).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)  # [co][ci][ky][kx]
    assert want[0, 0, 0, 0] == 0x3F80 and want[0, 1, 0, 0] == 0x3F82
    ref = want.reshape(64, 4, 2, 8, 9)  # [co][kc][chunk][i][tap]
    assert np.array_equal(packed.reshape(9, 4, 2, 64, 8), ref.transpose(4, 1, 2, 0, 3))
    assert h.afs_conv3x3_c64_pack_weights_bf16(None, packed.ctypes.data_as(ctypes.c_void_p)) == -1
