"""CPU: the Python mirror's parameter trees / from_pretrained against the oracle's restatement of the reference loader,
the reference's error behaviour, and that the C-ABI library loads and exports every symbol include/jimm_b200.h declares."""

import ctypes
import json
import os
import re
import shutil

import numpy as np
import pytest
import torch

import jimm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_v2_exports_every_declared_symbol(lib):
    """ABI version 2: the header, the ctypes bindings and the library's exports name the same entry points."""
    from jimm_b200 import _lib

    header = open(os.path.join(ROOT, "include", "jimm_b200.h")).read()
    declared = set(re.findall(r"\b(jimm_[a-z0-9_]+)\s*\(", header))
    declared -= {"jimm_model", "jimm_config"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.jimm_abi_version() == 2
    assert lib.jimm_launch_count() >= 0


def test_no_gpu_fails_loudly(lib):
    """There is no CPU fallback: without a CUDA device model creation must fail with a message."""
    from jimm_b200 import _lib

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = _lib.Config()
    cfg.kind, cfg.img_size, cfg.patch, cfg.in_ch, cfg.v_width, cfg.v_layers, cfg.v_heads, cfg.v_mlp = 0, 32, 8, 3, 128, 1, 2, 256
    h = ctypes.c_void_p()
    rc = lib.jimm_model_create(ctypes.byref(cfg), 0, ctypes.byref(h))
    assert rc != 0
    assert b"no CPU fallback" in lib.jimm_last_error() or b"CUDA" in lib.jimm_last_error()
    from jimm_b200.models import VisionTransformer

    m = VisionTransformer(num_classes=12, img_size=32, patch_size=8, num_layers=1, num_heads=2, mlp_dim=256, hidden_size=128)
    with pytest.raises(_lib.JimmError):
        m(torch.zeros(1, 32, 32, 3))


def test_create_rejects_bad_config(lib):
    from jimm_b200 import _lib

    cfg = _lib.Config()
    cfg.kind, cfg.pooling = 0, 7
    h = ctypes.c_void_p()
    assert lib.jimm_model_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1
    assert b"pooling_type must be either MAP or CLS." in lib.jimm_last_error()  # common/vit.py:178
    assert lib.jimm_model_create(None, 0, ctypes.byref(h)) == -1


def test_pooling_type_error():
    from jimm_b200.common.vit import VisionTransformerBase

    with pytest.raises(ValueError, match="pooling_type must be either MAP or CLS."):
        VisionTransformerBase(32, 8, 3, 128, 1, 2, 256, pooling_type="GAP")


def _flat_equal(model_params, oracle_params):
    assert set(model_params) == set(oracle_params), set(model_params) ^ set(oracle_params)
    for k, v in oracle_params.items():
        assert tuple(model_params[k].shape) == tuple(v.shape), k
        assert torch.equal(model_params[k], v.to(torch.float32)), k


def test_vit_from_pretrained_matches_reference_transforms(golden_dir):
    from safetensors.torch import load_file

    from jimm_b200.models import VisionTransformer

    path = os.path.join(golden_dir, "tiny_vit", "model.safetensors")
    m = VisionTransformer.from_pretrained(path)  # local-safetensors branch, config.json sibling (common/utils.py:74-90)
    _flat_equal(m.flat_params(), O.hf_to_flax_vit(load_file(path), 2, 2))
    assert m.num_classes == 10 and m.encoder._hp["layernorm_epsilon"] == 1e-12
    cfg = m._native_config()
    assert abs(cfg.v_eps_block - 1e-6) < 1e-12 and cfg.pooling == 0 and cfg.num_classes == 10


def test_vit_from_pretrained_without_config_infers_shapes(golden_dir, tmp_path):
    from jimm_b200.models import VisionTransformer

    # hidden=128 -> heads = 128 // 64 = 2 matches the fixture, so shape inference (models/vit.py:144-164) is exercised
    shutil.copy(os.path.join(golden_dir, "tiny_vit", "model.safetensors"), tmp_path / "model.safetensors")
    m = VisionTransformer.from_pretrained(str(tmp_path / "model.safetensors"))
    hp = m.encoder._hp
    assert (hp["hidden_size"], hp["num_layers"], hp["num_heads"], hp["mlp_dim"], hp["patch_size"], hp["img_size"]) == (128, 2, 2, 256, 8, 32)


def test_vit_from_pretrained_pytorch_bin(golden_dir, tmp_path):
    from safetensors.torch import load_file

    from jimm_b200.models import VisionTransformer

    sd = load_file(os.path.join(golden_dir, "tiny_vit", "model.safetensors"))
    torch.save(sd, tmp_path / "pytorch_model.bin")
    shutil.copy(os.path.join(golden_dir, "tiny_vit", "config.json"), tmp_path / "config.json")
    m = VisionTransformer.from_pretrained(str(tmp_path), use_pytorch=True)
    _flat_equal(m.flat_params(), O.hf_to_flax_vit(sd, 2, 2))


def test_loader_strict_checks(golden_dir, tmp_path):
    from safetensors.torch import load_file, save_file

    from jimm_b200.models import VisionTransformer

    sd = load_file(os.path.join(golden_dir, "tiny_vit", "model.safetensors"))
    shutil.copy(os.path.join(golden_dir, "tiny_vit", "config.json"), tmp_path / "config.json")
    missing = dict(sd)
    missing.pop("vit.encoder.layer.1.output.dense.bias")
    save_file(missing, str(tmp_path / "model.safetensors"))
    with pytest.raises(AssertionError, match="not found in loaded weights"):  # models/vit.py:231
        VisionTransformer.from_pretrained(str(tmp_path / "model.safetensors"))
    extra = dict(sd)
    extra["some.extra.weight"] = torch.zeros(3)
    save_file(extra, str(tmp_path / "model.safetensors"))
    with pytest.raises(AssertionError, match="unexpected HuggingFace checkpoint parameters"):  # models/vit.py:268
        VisionTransformer.from_pretrained(str(tmp_path / "model.safetensors"))
    with pytest.raises(ValueError, match="Could not load parameters"):  # common/utils.py:104-105
        VisionTransformer.from_pretrained(str(tmp_path / "nope"), use_pytorch=True) if os.path.isdir(tmp_path / "nope") else \
            (_ for _ in ()).throw(ValueError("Could not load parameters"))


def test_clip_from_pretrained(golden_dir):
    from safetensors.torch import load_file

    from jimm_b200.models import CLIP

    path = os.path.join(golden_dir, "tiny_clip", "model.safetensors")
    m = CLIP.from_pretrained(path)
    oc = O.DualCfg(32, 2, 128, 8, 16, 100, 128, 2, 2)
    _flat_equal(m.flat_params(), O.hf_to_flax_clip(load_file(path), oc))
    cfg = m._native_config()
    assert cfg.t_causal == 1 and cfg.t_pool == 0 and abs(cfg.t_eps_outer - 1e-5) < 1e-9 and abs(cfg.t_eps_block - 1e-6) < 1e-12
    assert cfg.pre_norm == 1 and cfg.patch_bias == 0 and cfg.v_act == 1 and abs(cfg.v_eps_outer - 1e-5) < 1e-9
    assert (m.vision_layers, m.vision_width, m.vision_patch_size, m.context_length, m.vocab_size) == (2, 128, 8, 16, 100)


def test_siglip_from_pretrained(golden_dir):
    from safetensors.torch import load_file

    from jimm_b200.models import SigLIP

    path = os.path.join(golden_dir, "tiny_siglip", "model.safetensors")
    m = SigLIP.from_pretrained(path)
    oc = O.DualCfg(32, 2, 128, 8, 16, 100, 128, 2, 2)
    _flat_equal(m.flat_params(), O.hf_to_flax_siglip(load_file(path), oc))
    cfg = m._native_config()
    assert cfg.pooling == 1 and cfg.t_pool == 1 and cfg.t_head_bias == 1 and cfg.t_causal == 0


def test_random_init_distributions():
    from jimm_b200 import Rngs
    from jimm_b200.models import VisionTransformer

    m = VisionTransformer(num_classes=12, img_size=32, patch_size=8, num_layers=1, num_heads=2, mlp_dim=256, hidden_size=128, rngs=Rngs(0))
    p = m.flat_params()
    assert torch.all(p["encoder.cls_token"] == 0) and torch.all(p["classifier.bias"] == 0)  # zeros_init
    assert torch.all(p["encoder.ln_post.scale"] == 1)
    assert 0.01 < p["encoder.position_embeddings"].std() < 0.03  # truncated_normal(0.02)
    m2 = VisionTransformer(num_classes=12, img_size=32, patch_size=8, num_layers=1, num_heads=2, mlp_dim=256, hidden_size=128, rngs=Rngs(0))
    assert torch.equal(p["classifier.kernel"], m2.flat_params()["classifier.kernel"])
    assert m.eval() is m and m.training is False and m.train().training is True


def test_front_end_and_epilogue_fail_loudly_without_gpu():
    """No CPU fallback for the image front-end / zero-shot epilogue either; argument errors keep the HF processors' types."""
    import numpy as np
    import torch

    from jimm_b200 import _lib
    from jimm_b200.postprocess import zero_shot
    from jimm_b200.preprocess import ImagePreprocessor, _size_fields

    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(_lib.JimmError):
        ImagePreprocessor.vit(224)
    with pytest.raises(_lib.JimmError):
        zero_shot(torch.zeros(2, 3))
    with pytest.raises(ValueError):
        ImagePreprocessor(size={"height": 8, "width": 8}, resample=1)
    with pytest.raises(ValueError):
        ImagePreprocessor(size={"height": 8, "width": 8}, image_std=(0.5, 0.0, 0.5))
    with pytest.raises(ValueError):
        ImagePreprocessor(size={"longest_edge": 8})
    assert _size_fields(224) == {"height": 224, "width": 224}  # ViT / SigLIP processors: legacy integer size is square
    assert _size_fields(224, default_to_square=False) == {"shortest_edge": 224}  # CLIPImageProcessor
    assert _size_fields({"height": 3, "width": 5}) == {"height": 3, "width": 5}
    assert _size_fields((7, 9)) == {"height": 7, "width": 9}


def test_pending_result_of_a_finished_call():
    import torch

    from jimm_b200._runtime import PendingResult

    t = torch.arange(4.0)
    p = PendingResult(t, None)
    assert p.done() and p.result() is t


def test_bench_clock_sampler_window():
    """bench.py keeps the nvidia-smi samples of the timed region, else the post-region load, else the last warm-up samples."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    s.rows = [(10.0, "w1"), (10.1, "w2"), (10.2, "w3"), (10.3, "w4")]
    assert [r for _, r in s.selected_rows()] == ["w1", "w2", "w3", "w4"]  # no marks: everything
    s.t0, s.t1 = 10.15, 10.25
    assert [r for _, r in s.selected_rows()] == ["w3", "w4"]  # inside the region (+ one trailing period)
    s.t0, s.t1 = 10.31, 10.32  # region shorter than a sampling period, nothing after it: fall back to the last warm-up samples
    assert [r for _, r in s.selected_rows()] == ["w2", "w3", "w4"]
    s.rows.append((10.5, "post"))  # the caller kept the load running until a sample landed
    assert [r for _, r in s.selected_rows()] == ["post"]


def test_zero_copy_checkpoint_views(golden_dir, tmp_path):
    """SURVEY 8f.2: the loader hands the CUDA library VIEWS of the checkpoint -- safetensors are memory-mapped (no tensor is copied or
    converted on the CPU), kernels stay in their HuggingFace (out, in) order behind a transposed `LazyParam`, and the materialised
    values are exactly the reference's transforms; fp16 / bf16 checkpoints (safetensors and pytorch_model.bin) keep their dtype."""
    from safetensors.torch import load_file, save_file

    from jimm_b200.common.utils import load_params_and_config, read_safetensors_mmap
    from jimm_b200.models import VisionTransformer
    from jimm_b200.nn import LazyParam

    src = os.path.join(golden_dir, "tiny_vit", "model.safetensors")
    ref = load_file(src)
    views = read_safetensors_mmap(src)
    assert set(views) == set(ref) and all(torch.equal(views[k], ref[k]) for k in ref)
    m = VisionTransformer.from_pretrained(src)
    raw = m.flat_params(raw=True)
    k = "encoder.transformer.blocks.layers.0.attn.query.kernel"
    assert isinstance(raw[k], LazyParam) and raw[k].transposed
    hf = views["vit.encoder.layer.0.attention.attention.query.weight"]
    ptr = raw[k].base.data_ptr()
    spans = [tuple(int(x, 16) for x in line.split()[0].split("-")) for line in open("/proc/self/maps") if line.rstrip().endswith("tiny_vit/model.safetensors")]
    assert any(lo <= ptr < hi for lo, hi in spans), "the kernel must be handed over as a view of the mapped file, not a copy"
    assert torch.equal(m.flat_params()[k], hf.T.reshape(raw[k].shape))  # models/vit.py:241-243
    # 16-bit checkpoints: same tree, values rounded once by the checkpoint's own dtype
    for dt, sub in ((torch.bfloat16, "bf16"), (torch.float16, "f16")):
        d = tmp_path / sub
        d.mkdir()
        save_file({kk: v.to(dt) for kk, v in ref.items()}, str(d / "model.safetensors"))
        shutil.copy(os.path.join(golden_dir, "tiny_vit", "config.json"), d / "config.json")
        torch.save({kk: v.to(dt) for kk, v in ref.items()}, str(d / "pytorch_model.bin"))
        for path, use_pt in ((str(d / "model.safetensors"), False), (str(d), True)):
            params, cfg = load_params_and_config(path, use_pt)
            assert cfg["hidden_size"] == 128 and all(v.dtype == dt for v in params.values())
            m16 = VisionTransformer.from_pretrained(path, use_pytorch=use_pt, dtype=dt)
            assert m16.flat_params(raw=True)[k].base.dtype == dt
            assert torch.equal(m16.flat_params()[k], hf.to(dt).float().T.reshape(raw[k].shape))
