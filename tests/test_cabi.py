"""CPU: the C-ABI library builds, loads and exports every symbol include/selfocc_b200.h declares."""
import os
import re
import subprocess
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, 'include', 'selfocc_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(so_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    from selfocc_b200 import build, _lib
    build.build()
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 12
    nm = subprocess.run(['nm', '-D', '--defined-only', _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(l.split()[-1] for l in nm.splitlines() if l.strip())
    for s in declared:
        assert s in exported, 'header declares %s but the library does not export it' % s
        assert s in _lib.SIGNATURES, 'ctypes binding lacks %s' % s
    assert sorted(_lib.SIGNATURES) == declared
    assert lib.so_abi_version() == _lib.ABI_VERSION
    assert lib.so_error_string(-1) == b'invalid argument'


def test_sm100a_only():
    from selfocc_b200 import _lib, build
    build.build()
    nvcc = build._nvcc()      # the toolkit that built the library; its bin/ need not be on PATH
    cuobjdump = os.path.join(os.path.dirname(nvcc), 'cuobjdump') if os.path.isabs(nvcc) else 'cuobjdump'
    out = subprocess.run([cuobjdump, '--list-elf', _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r'sm_\d+a?', out))
    assert archs == {'sm_100a'}, archs


def test_ops_refuse_cpu_tensors():
    import torch
    from selfocc_b200 import ops
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ops.msda_forward(torch.zeros(1, 4, 1, 16), torch.tensor([[2, 2]]), torch.tensor([0]),
                         torch.zeros(1, 1, 1, 1, 1, 2), torch.zeros(1, 1, 1, 1, 1))


def test_entry_points_reject_bad_arguments_without_a_gpu():
    """Error behaviour of the C ABI: null pointers / bad sizes return SO_ERR_INVALID_ARG (-1) or SO_ERR_UNSUPPORTED (-2)
    before any CUDA call is made, so this runs on a CPU-only box."""
    import ctypes as C
    from selfocc_b200 import _lib, build
    build.build()
    lib = _lib.load()
    N = None
    assert lib.so_msda_forward(N, N, N, N, N, N, 1, 1, 1, 16, 1, 1, 1, N) == -1
    assert lib.so_msda_backward(N, N, N, N, N, N, N, N, N, 1, 1, 1, 16, 1, 1, 1, N) == -1
    assert lib.so_linear_3xtf32(N, N, N, N, N, N, 10, 96, 96, 0, N) == -1
    one = C.c_void_p(16)   # non-null, 16-byte aligned dummy (never dereferenced on these paths)
    assert lib.so_linear_3xtf32(one, one, one, N, N, one, 10, 96, 100, 0, N) == -2      # K not a multiple of 96
    assert lib.so_linear_3xtf32(one, one, one, N, N, one, 0, 96, 96, 0, N) == 0         # M = 0: nothing to do
    assert lib.so_layer_norm(N, N, N, N, N, 4, 96, 1e-5, N) == -1
    assert lib.so_layer_norm(one, N, one, one, one, 4, 1000, 1e-5, N) == -2
    assert lib.so_point_sampling(N, N, 1, 1, 1, 1.0, 1.0, N, N, N, N) == -1
    assert lib.so_render_infer(N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N) == -1
    d = _lib.VolumeDesc()
    d.H, d.W, d.Z, d.zpitch = 4, 4, 4, 2            # zpitch < Z
    assert lib.so_field_query(one, N, C.byref(d), one, 1, one, N, N, N) == -1
    assert lib.so_tpv_decode(one, one, one, 48, one, one, one, one, C.byref(d), one, N, N) == -1   # invalid volume desc
    big = _lib.VolumeDesc()
    big.H, big.W, big.Z, big.zpitch = 40000, 40000, 2, 8          # > 2^31 sdf entries: the kernels index with 32 bits
    for i in range(3):
        big.axis[i].range0, big.axis[i].size0 = 1.0, 1.0
    assert lib.so_field_query(one, N, C.byref(big), one, 1, one, N, N, N) == -2
    assert lib.so_render_train_pair_floats(C.byref(big)) == 0 and lib.so_render_train_pair_floats(None) == 0
    ok = _lib.VolumeDesc()
    ok.H, ok.W, ok.Z, ok.zpitch = 257, 257, 31, 32
    for i in range(3):
        ok.axis[i].range0, ok.axis[i].size0 = 51.2, 128.0
    assert lib.so_render_train_pair_floats(C.byref(ok)) == 2 * 257 * 257 * 32
    # training forward: a mis-aligned pair scratch is refused before any launch
    assert lib.so_render_train_forward(one, N, C.byref(ok), one, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, one,
                                       C.c_void_p(20), N) == -1
    assert lib.so_error_string(-2) == b'unsupported configuration'
    assert lib.so_render_workspace_floats(0) == 2 and lib.so_render_workspace_floats(24) == 48
    # ---- round-2 entry points
    assert lib.so_render_pack_floats(None) == 0 and lib.so_render_pack_floats(C.byref(big)) == 0
    assert lib.so_render_pack_floats(C.byref(ok)) == 2 * 257 * 257 * 32            # n_feat 0: float2 z-pairs
    ok3 = _lib.VolumeDesc()
    ok3.H, ok3.W, ok3.Z, ok3.zpitch, ok3.n_feat, ok3.feat_pitch = 257, 257, 31, 32, 3, 4
    for i in range(3):
        ok3.axis[i].range0, ok3.axis[i].size0 = 51.2, 128.0
    assert lib.so_render_pack_floats(C.byref(ok3)) == 4 * 257 * 257 * 31           # n_feat 3: float4 (r, g, b, sdf)
    ok8 = _lib.VolumeDesc()
    ok8.H, ok8.W, ok8.Z, ok8.zpitch, ok8.n_feat, ok8.feat_pitch = 9, 9, 5, 8, 8, 8
    for i in range(3):
        ok8.axis[i].range0, ok8.axis[i].size0 = 1.0, 4.0
    assert lib.so_render_pack_floats(C.byref(ok8)) == 0                            # no packed form for 8 channels
    assert lib.so_render_pack(one, N, C.byref(ok8), one, N) == -2
    assert lib.so_render_pack(N, N, C.byref(ok), one, N) == -1
    assert lib.so_render_pack(one, N, C.byref(ok3), one, N) == -1                  # colour pack without a feature volume
    assert lib.so_render_infer_packed(N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N, N) == -1
    assert lib.so_tpv_decode_rows(one, one, one, 96, one, one, one, one, C.byref(ok), 250, 10, one, N, N) == -1   # rows beyond H
    assert lib.so_tpv_decode_rows(one, one, one, 96, one, one, one, one, C.byref(ok), 7, 0, one, N, N) == 0       # empty slab
    assert lib.so_field_second_grad(N, C.byref(ok), one, 1, one, N) == -1
    assert lib.so_field_second_grad(one, C.byref(ok), one, 0, one, N) == 0
    assert lib.so_field_second_grad_backward(C.byref(ok), one, 1, N, one, N) == -1
    assert lib.so_depth_metric_sample(N, one, 1, 1, 1, 1, one, N) == -1
    assert lib.so_depth_metric_sample(one, one, 6, 0, 45, 80, one, N) == 0          # no LiDAR points: nothing to do
    assert lib.so_depth_metric_sums(one, one, N, N, 6, 10, one, N) == -1
    assert lib.so_flatten_level(one, one, one, one, 6, 96, 100, 50, 120, N) == -1   # level does not fit the token tensor
    assert lib.so_flatten_level(N, one, one, one, 6, 96, 100, 0, 100, N) == -1
    # decode backward slab kernels
    assert lib.so_tpv_decode_bwd_features(N, one, one, 96, C.byref(ok), 0, 8, one, N) == -1
    assert lib.so_tpv_decode_bwd_features(one, one, one, 96, C.byref(ok), 250, 10, one, N) == -1      # rows beyond H
    assert lib.so_tpv_decode_bwd_features(one, one, one, 94, C.byref(ok), 0, 8, one, N) == -2         # C not a multiple of 4
    assert lib.so_tpv_decode_bwd_features(one, one, one, 96, C.byref(ok), 7, 0, one, N) == 0          # empty slab
    assert lib.so_tpv_decode_bwd_hidden(one, N, N, N, 96, C.byref(ok), 0, 8, one, one, N) == -1
    assert lib.so_tpv_decode_bwd_hidden(one, N, N, one, 96, C.byref(ok), 0, 8, C.c_void_p(20), one, N) == -1   # mis-aligned g1
    assert lib.so_tpv_decode_bwd_input(one, one, 6, N) == -1 and lib.so_tpv_decode_bwd_input(one, one, 0, N) == 0
    # strided attention entry points: odd offset pitch / mis-aligned offsets are refused (float2 loads)
    assert lib.so_tpv_self_attn_forward_strided(one, one, one, one, one, one, one, 10, 6, 16, 4, 3, 4, 96, 6 * 3 * 4 * 2 + 1, 6 * 3 * 4, N) == -1
    assert lib.so_tpv_self_attn_forward_strided(one, one, one, C.c_void_p(20), one, one, one, 10, 6, 16, 4, 3, 4, 96, 6 * 3 * 4 * 2, 6 * 3 * 4, N) == -1
    for hook in (lib.so_attn_force_v1, lib.so_linear_force_ss, lib.so_render_train_force_sem_generic):
        assert hook(1) == 0 and hook(0) == 0


def test_product_never_imports_the_oracle_or_reads_the_reference():
    """The oracle is test infrastructure: only tests/, smoke() and bench.py's CPU legs may touch it, and nothing that
    ships may read /root/reference at run time."""
    import os, re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, 'selfocc_b200')
    bad = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith(('.py', '.cu', '.cuh', '.h')):
                continue
            text = open(os.path.join(dirpath, f), errors='ignore').read()
            if re.search(r'^\s*(from|import)\s+oracle\b', text, re.M) or '/root/reference' in text:
                bad.append(os.path.relpath(os.path.join(dirpath, f), root))
    assert not bad, bad
    for f in ('bench.py', '__graft_entry__.py'):
        assert '/root/reference' not in open(os.path.join(root, f)).read(), f


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No silent fallback: a missing libselfocc_b200.so is an error at the first op, not a slower path."""
    from selfocc_b200 import _lib
    monkeypatch.setattr(_lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    monkeypatch.setattr(_lib, '_lib', None)
    with pytest.raises(_lib.SelfOccLibraryError):
        _lib.load()
