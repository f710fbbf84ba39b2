"""CPU suite: the C-ABI library loads without a GPU and exports every symbol include/inerf_b200.h declares;
argument validation returns error codes instead of launching.  No compute calls here."""
import ctypes
import os
import re

import pytest

from instance_nerf_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def test_header_symbols_all_exported(L):
    hdr = open(os.path.join(ROOT, "include", "inerf_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(inerf_[A-Za-z0-9_]+)\s*\(", hdr)))
    assert declared, "no declarations parsed"
    missing = [s for s in declared if not hasattr(L, s)]
    assert not missing, f"declared in the header but not exported: {missing}"
    assert sorted(declared) == sorted(_lib.EXPORTED_SYMBOLS), "ctypes prototypes and the header disagree"


def test_version_and_error_strings(L):
    assert L.inerf_version() >= 1000
    assert L.inerf_error_string(0) == b"ok"
    for code in (-1, -2, -3, -4, -5):
        assert L.inerf_error_string(code).startswith(b"inerf:")


def test_bad_arguments_return_codes_without_a_gpu(L):
    # NULL pointers / bad sizes are rejected before any launch (the reference's raymarching ops check nothing)
    assert L.inerf_near_far_from_aabb(None, None, None, 4, 0.2, None, None, None) == -1
    assert L.inerf_grid_encode_forward(None, None, None, None, 8, 3, 2, 16, 1.0, 16, None, 0, 0, 0, 0, 1, None) < 0
    assert L.inerf_field_weights_bytes(0) == 0 and L.inerf_field_weights_bytes(65) == 0
    assert L.inerf_field_weights_bytes(32) == (64 * 32 + 16 * 64 + 64 * 32 + 64 * 64 + 16 * 64 + 64 * 48 + 64 * 64 + 32 * 64) * 2
    assert L.inerf_render_fused(None, None, None, None, None, None, 1, 4, 128, 0.0, 1024, 1e-4, None, None, None, None, None, None) < 0


def test_pack_weights_layout_roundtrip(L):
    """Host-side packing into the UMMA K-major core-matrix layout: element (n, k) of a layer lands at
    (n%8)*16 + (n/8)*SBO + (k/8)*128 + (k%8)*2 with SBO = (Kpad/8)*128 (csrc/umma.cuh)."""
    import numpy as np
    K = 5
    rng = np.random.RandomState(0)
    shapes = [(64, 32), (16, 64), (64, 31), (64, 64), (3, 64), (64, 47), (64, 64), (K, 64)]
    ws = [np.ascontiguousarray(rng.randn(*s).astype(np.float32)) for s in shapes]
    n = L.inerf_field_weights_bytes(K)
    blob = np.zeros(n, np.uint8)
    rc = L.inerf_field_pack_weights(*[w.ctypes.data for w in ws], K, blob.ctypes.data)
    assert rc == 0
    h = blob.view(np.float16)
    pads = [(64, 32), (16, 64), (64, 32), (64, 64), (16, 64), (64, 48), (64, 64), (16, 64)]
    base = 0
    for w, (Np, Kp) in zip(ws, pads):
        sbo = (Kp // 8) * 128
        for (r, c) in [(0, 0), (w.shape[0] - 1, w.shape[1] - 1), (w.shape[0] // 2, 7), (1, 8)]:
            off = base + (r % 8) * 16 + (r // 8) * sbo + (c // 8) * 128 + (c % 8) * 2
            assert h[off // 2] == np.float16(w[r, c])
        base += Np * Kp * 2
    assert base == n


@pytest.mark.parametrize("K", [5, 16, 64])
def test_pack_weights_bwd_layout(L, K):
    """Host-side packing of the mask-head backward blob, every byte: five [Npad x Kpad] K-major tiles, element (n, k) at
    the same offset as in the forward round trip.  W0, W1 as they are; W2, W1, W0[:, :32] transposed, (n, k) = W[k][n],
    with zeros where the output index k >= K (W2) and in every padding row or column."""
    import numpy as np
    rng = np.random.RandomState(1)
    m0, m1, m2 = (np.ascontiguousarray(rng.randn(*s).astype(np.float32)) for s in [(64, 47), (64, 64), (K, 64)])
    n = L.inerf_field_bwd_weights_bytes()
    blob = np.full(n, 0xA5, np.uint8)   # not zero: the packer must write every byte
    assert L.inerf_field_pack_weights_bwd(m0.ctypes.data, m1.ctypes.data, m2.ctypes.data, K, blob.ctypes.data) == 0
    h = blob.view(np.float16)
    base = 0
    for i, (src, Np, Kp) in enumerate([(m0, 64, 48), (m1, 64, 64), (m2.T, 64, 64), (m1.T, 64, 64), (m0.T, 32, 64)]):
        n_, k_ = np.meshgrid(np.arange(Np), np.arange(Kp), indexing="ij")
        got = h[base // 2 + ((n_ % 8) * 16 + (n_ // 8) * ((Kp // 8) * 128) + (k_ // 8) * 128 + (k_ % 8) * 2) // 2]
        want = np.zeros((Np, Kp), np.float16)
        r, c = min(Np, src.shape[0]), min(Kp, src.shape[1])
        want[:r, :c] = src[:r, :c]
        assert np.array_equal(got.view(np.uint16), want.view(np.uint16))
        if i == 2:
            assert not np.any(got[:, K:])   # transposed W2: output index o >= K is zero
        base += Np * Kp * 2
    assert base == n
    assert L.inerf_field_pack_weights_bwd(m0.ctypes.data, m1.ctypes.data, m2.ctypes.data, 0, blob.ctypes.data) == -2
    assert L.inerf_field_pack_weights_bwd(None, m1.ctypes.data, m2.ctypes.data, K, blob.ctypes.data) == -1


def test_product_path_has_no_cpu_fallback():
    import torch
    from instance_nerf_b200 import raymarching
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(Exception):
        raymarching.composite_rays_train(torch.zeros(4), torch.zeros(4, 3), torch.zeros(4, 2), torch.zeros(1, 3, dtype=torch.int32))


def test_reference_packages_import_with_backend_shims():
    """Drop-in check at the reference's own import site (needs /root/reference: this container only).  The reference's
    op packages do `import _raymarching as _backend` etc.; with our shims registered under those names the reference's
    wrappers import unchanged and see every function they call."""
    import sys
    ref_root = "/root/reference/instance_nerf"
    if not os.path.isdir(ref_root):
        pytest.skip("/root/reference not present (GPU box)")
    import importlib
    import instance_nerf_b200.backend as b
    saved = {k: sys.modules.get(k) for k in ("_raymarching", "_gridencoder", "_shencoder", "raymarching", "gridencoder", "shencoder")}
    sys.modules["_raymarching"], sys.modules["_gridencoder"], sys.modules["_shencoder"] = b.raymarching, b.gridencoder, b.shencoder
    for k in ("raymarching", "gridencoder", "shencoder"):
        sys.modules.pop(k, None)
    sys.path.insert(0, ref_root)
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            rm = importlib.import_module("raymarching")
            ge = importlib.import_module("gridencoder")
            sh = importlib.import_module("shencoder")
        assert rm.raymarching._backend is b.raymarching and ge.grid._backend is b.gridencoder and sh.sphere_harmonics._backend is b.shencoder
        src = open(os.path.join(ref_root, "raymarching", "raymarching.py")).read()
        used = set(re.findall(r"_backend\.([A-Za-z0-9_]+)\(", src))
        assert used and used <= set(vars(b.raymarching)), used - set(vars(b.raymarching))
        src = open(os.path.join(ref_root, "gridencoder", "grid.py")).read()
        assert set(re.findall(r"_backend\.([A-Za-z0-9_]+)\(", src)) <= set(vars(b.gridencoder))
        src = open(os.path.join(ref_root, "shencoder", "sphere_harmonics.py")).read()
        assert set(re.findall(r"_backend\.([A-Za-z0-9_]+)\(", src)) <= set(vars(b.shencoder))
    finally:
        sys.path.remove(ref_root)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_new_entry_points_reject_bad_arguments_without_a_gpu(L):
    """Argument validation of the entry points added for the single-walk marcher and the fused optimizer step."""
    assert L.inerf_march_scratch_floats(4096, 1024) == 4096 * 1024 and L.inerf_march_scratch_floats(0, 1024) == 0
    # C = 0 / non power-of-two H are rejected before any launch
    assert L.inerf_march_rays_train_count_t(None, None, None, 8.0, 0.0, 1024, 16, 0, 128, None, None, None, None, None, None, None) < 0
    assert L.inerf_march_rays_train_expand(None, None, 8.0, 0.0, 1024, 16, 4, 100, 64, None, None, None, None, None, None, None, None) < 0
    # NULL tensors with n > 0
    assert L.inerf_adam_step(None, None, None, None, 8, 1e-2, 0.9, 0.99, 1e-15, None, None, None, 1.0, None) == -1
    assert L.inerf_adam_advance(None, None, None) == -1
    # n == 0 is a no-op
    assert L.inerf_adam_step(None, None, None, None, 0, 1e-2, 0.9, 0.99, 1e-15, None, None, None, 1.0, None) == 0


def test_field_desc_struct_matches_header():
    """ctypes mirror of struct inerf_field_desc: field order / types as declared in include/inerf_b200.h."""
    hdr = open(os.path.join(ROOT, "include", "inerf_b200.h")).read()
    body = re.search(r"typedef struct inerf_field_desc \{(.*?)\} inerf_field_desc;", hdr, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*;", body)
    assert names == [f[0] for f in _lib.FieldDesc._fields_]
    assert ctypes.sizeof(_lib.FieldDesc) == 3 * 8 + 6 * 4 + 8   # 3 pointers, 6 x 32-bit, 1 pointer (no padding)


def test_bench_reference_arm_prints_exactly_one_json_line():
    """bench.py's contract: ONE JSON line on stdout (library banners are redirected to stderr); the CPU reference arm runs
    without a GPU, on a bounded sample."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "Mrays/s" and j["value"] > 0 and j["gpu_launches"] == 0
    assert j["cpu_baseline"]["kind"] == "port" and j["e2e"]["h2d_bytes_per_step"] == 0
