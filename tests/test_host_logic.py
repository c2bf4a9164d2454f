"""CPU tests of the host side: the Keras weight table, initialisers, the builder helpers, and that the
C-ABI library loads and exports every symbol include/vitdet_b200.h declares (no compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest

from _util import ROOT, oracle, tiny_config
import vision_transformer_detector_b200 as vd
from vision_transformer_detector_b200 import _capi, keras_init


def test_weight_table_matches_oracle_restatement():
    for cfg in (vd.DetectorConfig(), tiny_config(),
                vd.DetectorConfig(input_shape=(640, 640, 3), patch_size=16, embedding_dim=768, encoder_num_heads=12,
                                  encoder_key_dim=64, encoder_repeat_times=12, encoder_mlp_quantities=3),
                tiny_config(mlp_head_dense_mish_block_repeats=2)):
        assert vd.weight_specs(cfg) == oracle.weight_table(cfg)


def test_default_model_size():
    specs = vd.weight_specs(vd.DetectorConfig())
    assert len(specs) == 245                                     # notebook cell 7 progress bar "…/245"
    assert sum(int(np.prod(s)) for _, s in specs) == 131_476_891


def test_keras_initialisers():
    rng = np.random.default_rng(0)
    assert keras_init.compute_fans((28, 8, 40)) == (224.0, 1120.0)       # limit sqrt(6/1344)
    assert keras_init.compute_fans((8, 40, 28)) == (320.0, 224.0)        # limit sqrt(6/544)
    k = keras_init.init_weight(rng, "multi_head_attention/query/kernel", (28, 8, 40))
    assert k.dtype == np.float32 and np.abs(k).max() <= np.sqrt(6 / 1344) and np.abs(k).max() > 0.9 * np.sqrt(6 / 1344)
    assert not keras_init.init_weight(rng, "dense/bias", (17,)).any()
    assert (keras_init.init_weight(rng, "layer_normalization/gamma", (28,)) == 1).all()
    e = keras_init.init_weight(rng, "position_encoding/position_embedding/embeddings", (1296, 1))
    assert np.abs(e).max() <= 0.05


def test_builder_helpers_mirror_the_reference_signatures():
    x = vd.vision_transformer_detector.Input((608, 608, 3))
    e = vd.transformer_preprocessor(x, patch_size=17, embedding_dim=28, max_weight=10, clip_weight=True)
    assert e.shape == (None, 1296, 28)
    enc = vd.transformer_encoder(e, use_mish=True, num_heads=8, key_dim=40, dropout=None, mlp_quantities=8,
                                 repeat_times=8, max_weight=10, clip_weight=True)
    assert enc.shape == (None, 1296, 28)
    h = vd.mlp_head(enc, use_mish=True, mlp_head_last_units=136, dense_layers_quantity=7, dense_mish_block_repeats=1,
                    dropout=None, max_weight=10, clip_weight=True)
    assert h.shape == (None, 17, 6)
    with pytest.raises(NotImplementedError):
        vd.transformer_encoder(e, use_mish=True, num_heads=8, key_dim=40, dropout=0.1, mlp_quantities=8,
                               repeat_times=8, max_weight=10, clip_weight=True)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "vitdet_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(vitdet_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_capi.lib_path())
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/vitdet_b200.h but not exported"
    assert declared == set(_capi.SYMBOLS), "ctypes table and header disagree"
    assert _capi.load().vitdet_abi_version() == 2


def test_struct_layouts_match_the_header():
    assert ctypes.sizeof(_capi.Config) == 15 * 4
    assert ctypes.sizeof(_capi.DecodeParams) == 8 * 4
    assert ctypes.sizeof(_capi.Detections) == 6 * ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(_capi.DenseEx) == 56
    c = _capi.default_config()
    assert (c.image_h, c.image_w, c.patch_size, c.embedding_dim, c.num_heads, c.key_dim) == (608, 608, 17, 28, 8, 40)
    assert (c.mlp_quantities, c.repeat_times, c.head_last_units, c.head_dense_layers, c.head_block_repeats) == (8, 8, 136, 7, 1)
    assert (c.use_mish, c.num_slots, c.classes) == (1, 17, 80) and abs(c.ln_epsilon - 1e-3) < 1e-9


def test_no_cpu_fallback():
    """Without a CUDA device the product must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(_capi.VitdetError) as ei:
        vd.create_vision_transformer_detector()
    assert ei.value.code == _capi.E_NO_DEVICE
    with pytest.raises(_capi.VitdetError):
        vd.transform_predictions(np.zeros((1, 17, 6), np.float32))


def test_metric_class_mirrors_the_reference_interface():
    """MeanAveragePrecision (det.py:1268-2060): same constructor default, method names and update_state signature;
    without a GPU it fails loudly instead of computing on the host."""
    import inspect
    import torch
    m = vd.MeanAveragePrecision
    sig = inspect.signature(m.update_state)
    assert list(sig.parameters)[:5] == ["self", "y_true", "y_pred", "sample_weight", "use_transform_predictions"]
    assert sig.parameters["sample_weight"].default is None and sig.parameters["use_transform_predictions"].default is True
    assert inspect.signature(m.__init__).parameters["name"].default == "AP"
    for attr in ("result", "reset_state", "latest_positive_bboxes", "labels_quantity_per_image", "showed_up_classes"):
        assert hasattr(m, attr)
    assert (vd.Constants.LATEST_RELATED_IMAGES.value, vd.Constants.BBOXES_PER_IMAGE.value) == (3, 14)     # det.py:32, 37
    if not torch.cuda.is_available():
        with pytest.raises(_capi.VitdetError) as ei:
            m()
        assert ei.value.code == _capi.E_NO_DEVICE


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "vision_transformer_detector_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "vitdet_oracle" not in text and "import oracle" not in text and "import map_oracle" not in text, \
                    f"{f} references the oracle"


def test_category_names_match_the_reference_table():
    """tests/golden/coco_categories.csv: the 80 categories of the COCO 2017 instance annotations (id and name as in their
    `categories` list), numbered 0..79 in ascending COCO id, which is the reference's `id_in_model` order
    (full_categories.csv)."""
    path = os.path.join(ROOT, "tests", "golden", "coco_categories.csv")
    assert len(vd.COCO_CATEGORY_NAMES) == 80 and vd.COCO_CATEGORY_NAMES[0] == "person" and vd.COCO_CATEGORY_NAMES[79] == "toothbrush"
    import csv
    rows = list(csv.DictReader(open(path)))
    assert [int(r["id_in_coco"]) for r in sorted(rows, key=lambda r: int(r["id_in_model"]))] == sorted(int(r["id_in_coco"]) for r in rows)
    assert [r["name"] for r in sorted(rows, key=lambda r: float(r["id_in_model"]))] == list(vd.COCO_CATEGORY_NAMES)


def test_traffic_capture_is_stamped_for_the_current_kernel_sources():
    """bench.py quotes roofline.traffic from profiles/gemm_mlp_2_traffic.json only while the capture's stamp equals the hash
    of the dominant kernel's SASS (gemm_tc_kernel<ACT_MISH, 0, false, true>, the CTA-pair bf16 Mish instance, compiled
    with the library's nvcc flags).  A change to its machine code needs a new `ncu --set full` capture
    (scripts/gpu_round2.sh + scripts/summarize_profiles.py), otherwise the bench line silently carries `traffic: null`."""
    import json
    import os
    from vision_transformer_detector_b200 import build
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "gemm_mlp_2_traffic.json")
    t = json.load(open(path))
    assert t["kernel_hash"] == build.kernel_hash(), "re-capture the dominant GEMM under ncu: its machine code changed"
    assert t["rows_per_launch"] == 64 * 1296
    # no re-reads: measured DRAM traffic within 5 % of the algorithmic bytes 2 (M (K + N) + K N)
    algorithmic = 2.0 * (82944 * (3584 + 1792) + 3584 * 1792)
    assert 0.9 * algorithmic < t["traffic_bytes_per_launch"] < 1.05 * algorithmic
