"""CPU-side checks of the drop-in boundary: libb2r.so loads without a GPU, exports every symbol
include/b2r.h declares, and the ctypes table covers exactly those symbols; argument validation of
the entry points that need no device work."""
import ctypes as C
import os
import re

import pytest

from msra_practice_project_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "b2r.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2r_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    syms = header_symbols()
    assert len(syms) >= 15
    lib = _lib.lib()
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/b2r.h but not exported by libb2r.so"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes table and header disagree"


def test_version_and_size_queries():
    lib = _lib.lib()
    assert lib.b2r_version() == 100
    assert lib.b2r_mlp_tc_packed_bytes(0) > 1187840
    assert lib.b2r_mlp_f32_workspace_bytes(0, 10, 1) == 10 * 2516 * 4
    assert lib.b2r_mlp_f32_workspace_bytes(1, 10, 1) == 10 * 4616 * 4
    assert lib.b2r_mlp_f32_workspace_bytes(0, 10 ** 7, 0) == 65536 * 2516 * 4      # inference is chunked
    assert lib.b2r_mlp_f32_bwd_scratch_bytes(0, 3) == 3 * 512 * 4


def test_bad_arguments_return_negative_and_set_message():
    lib = _lib.lib()
    rc = lib.b2r_composite_fwd(None, None, None, 3, 1, 1, None, None, None, None, None)
    assert rc < 0 and b"NULL" in lib.b2r_last_error()
    rc = lib.b2r_sample_pdf(None, 0, None, 0, None, 1, 4, 4, None, 0, None, None, None, None)
    assert rc < 0
    inp = _lib.MlpInput()
    rc = lib.b2r_mlp_tc_fwd(0, 16, 1, C.byref(inp), 16, 0, None, None)
    assert rc < 0 and b"exactly one" in lib.b2r_last_error()
    with pytest.raises(RuntimeError):
        _lib.check(rc, "b2r_mlp_tc_fwd")
    # the layer-wise path has two GEMM engines, 0 (fp32) and 1 (tf32); gemm_mode is checked before anything else (the calls
    # below would otherwise fail on the 64-byte workspace / on having nothing to differentiate)
    inp.x, inp.n_rays, inp.n_samples = 256, 512, 1
    assert lib.b2r_mlp_f32_fwd(0, 16, None, 1, C.byref(inp), 16, 16, 64, 1, 2, None) < 0 and b"gemm_mode" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_bwd(0, 16, None, 1, C.byref(inp), 16, 16, 16, 16, 1 << 30, None, None, 2, None) < 0 \
        and b"gemm_mode" in lib.b2r_last_error()


def test_grad_precision_names():
    """One engine per gradient precision: fp32 / tf32 = the layer-wise path, bf16 (default) = the fused training path."""
    from msra_practice_project_b200 import ops
    assert ops.get_grad_precision() == "bf16"
    with pytest.raises(ValueError):
        ops.set_grad_precision("auto")
    assert ops.get_grad_precision() == "bf16"


def test_training_and_batched_entry_points_sizes_and_argument_checks():
    """Size queries and argument validation of the entry points added for training / batched latents / SirenNeRF."""
    lib = _lib.lib()
    # 1000 rows -> 4 tiles of 256 -> 2 tile pairs -> 8 sub-tiles of 128 rows
    per_sub_saved = 40 * 16384 + 8 * 2 * 128 * 16 + 2 * 128 * 8
    assert lib.b2r_mlp_tc_train_saved_bytes(0, 1000) == 8 * per_sub_saved
    assert lib.b2r_mlp_tc_train_scratch_bytes(0, 1000) == 8 * (38 * 16384 + 128 * 16)
    assert lib.b2r_mlp_tc_train_saved_bytes(3, 1000) == 0 and lib.b2r_mlp_tc_train_saved_bytes(0, 0) == 0
    assert lib.b2r_mlp_tc_bwd_packed_bytes(0) == 34 * 32768 + 640 * 4 and lib.b2r_mlp_tc_bwd_packed_bytes(3) == 0
    # FiLM-SIREN: 37 tile blocks + 9 layers of thread-major cosine bytes per sub-tile; 36 gradient blocks + head gradients
    assert lib.b2r_mlp_tc_train_saved_bytes(1, 1000) == 8 * (37 * 16384 + 9 * 32768)
    assert lib.b2r_mlp_tc_train_scratch_bytes(1, 1000) == 8 * (36 * 16384 + 128 * 16)
    assert lib.b2r_mlp_tc_bwd_packed_bytes(1) == 32 * 32768 + 1024 * 4
    # chunk area + fp32 tables + the inference kernels' blobs [h chunk 3 | compact post chunk] per step and N-half (tc_core.cuh extra_base)
    assert lib.b2r_mlp_tc_packed_bytes(1) == 8 * 5 * 32768 + 2308 * 4 + 8 * 2 * (16384 + 4096)            # FiLM-SIREN
    assert lib.b2r_mlp_tc_packed_bytes(2) == 8 * 5 * 32768 + 5 * 16384 + 1668 * 4 + 8 * 2 * (16384 + 4096) + 2 * (8192 + 2048)      # SirenNeRF
    assert lib.b2r_mlp_f32_workspace_bytes(2, 10, 1) == 10 * 4620 * 4
    inp = _lib.MlpInput()
    inp.x, inp.n_rays, inp.n_samples = 256, 512, 1
    assert lib.b2r_mlp_tc_train_fwd(3, 16, C.byref(inp), 16, 16, 1 << 30, None, None) < 0 and b"unknown model kind" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_bwd(1, 16, 512, 16, 16, 16, 16, 1 << 30, 16, None) < 0 and b"NeRF" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_pack_bwd_film(None, None, 1, 1, 16, None) < 0
    assert lib.b2r_mlp_tc_train_bwd_film(16, 16, 16, 1, 1, 0, 512, 16, 16, 16, 16, 64, 16, 16, 16, None) < 0 and b"scratch" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_bwd_film(16, 16, 16, 0, 2, 256, 512, 16, 16, 16, 16, 1 << 30, 16, 16, 16, None) < 0 and b"multiple of 512" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_fwd_film_batched(16, 2, 256, C.byref(inp), 16, 16, 1 << 30, None, None) < 0 and b"multiple of 512" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_fwd(0, 16, C.byref(inp), 16, 16, 64, None, None) < 0 and b"too small" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_bwd(0, 16, 512, 16, 16, 16, 16, 64, 16, None) < 0 and b"scratch" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_fwd_film_batched(16, 2, 100, C.byref(inp), 16, 0, None, None) < 0 and b"multiple of 512" in lib.b2r_last_error()
    inp.n_rays = 1024
    assert lib.b2r_mlp_tc_fwd_film_batched(16, 1, 512, C.byref(inp), 16, 0, None, None) < 0 and b"latents" in lib.b2r_last_error()
    # last-sample sign check (b2r_last_sample): argument validation of the kernels that flag and of the fp32 re-evaluation
    ls = _lib.LastSample(64, 8, None, None, 0.01, 0.0)
    assert lib.b2r_mlp_tc_fwd(0, 16, 1, C.byref(inp), 16, 0, C.byref(ls), None) < 0 and b"count / ray_ids" in lib.b2r_last_error()
    rin = _lib.MlpInput()
    rin.rays, rin.z, rin.n_rays, rin.n_samples = 256, 256, 8, 64
    ls = _lib.LastSample(32, 8, 16, 16, 0.01, 0.0)
    assert lib.b2r_mlp_tc_fwd(0, 16, 1, C.byref(rin), 16, 0, C.byref(ls), None) < 0 and b"samples_per_ray" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_last_sigma(0, 16, None, 1, 1, 0, C.byref(rin), 32, 16, 4, 16, 16, 1 << 30, None) < 0 and b"samples_per_ray" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_last_sigma(0, 16, None, 1, 1, 0, C.byref(rin), 64, 16, 4, 16, 16, 64, None) < 0 and b"workspace too small" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_last_sigma(1, 16, None, 1, 1, 0, C.byref(rin), 64, 16, 4, 16, 16, 1 << 30, None) < 0 and b"film" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_last_sigma(0, 16, None, 1, 1, 0, C.byref(rin), 64, 16, 0, 16, 16, 1 << 30, None) == 0          # nothing flagged
    assert lib.b2r_mlp_tc_pack_film_batched(None, None, 1, 2, None, None) < 0
    assert lib.b2r_adam_step(None, None, None, None, 4, None, 1e-3, 0.1, 0.0, 0.9, 0.999, 1e-8, 1.0, None) < 0
    assert lib.b2r_to8b(None, 4, None, None) < 0 and lib.b2r_to8b(None, 0, None, None) == 0
