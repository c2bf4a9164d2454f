"""GPU parity tests of the PRODUCT (bf16) kernels against a bf16-faithful oracle.

The 2e-2 tolerance north_star allows the bf16 mode against the float64 reference is dominated by the rounding of the
operands to bf16 — which is the same for a correct and for a subtly wrong kernel.  Here the oracle rounds exactly where
the kernels round (oracle.bf16_round / forward_bf16: operands and stored activations in bf16, accumulation in float64),
so what is left is accumulation order, ex2/rcp.approx and one-ulp rounding flips: a dropped k-tail, a wrong swizzle
column, a mis-fused LayerNorm or cross-image leakage in the last key tile is orders of magnitude above that.  Every
tensor-core kernel the benchmark times is covered at operator level (both GEMM kernels with both epilogues, the fused
LayerNorm / position-add epilogues, the fused MLP tail, the slot projection, all three attention kernels), then the
whole model, fused against unfused builds, and batch independence.
"""

import numpy as np
import pytest

from _util import build_model, images, oracle, rel_err, tiny_config
import vision_transformer_detector_b200 as vd

pytestmark = pytest.mark.gpu



def bf16_ulp(x):
    """Spacing of bfloat16 (8 significand bits) at |x|: 2^(floor(log2|x|) - 7)."""
    ax = np.maximum(np.abs(np.asarray(x, np.float64)), 2.0 ** -120)
    return 2.0 ** (np.floor(np.log2(ax)) - 7)


R = oracle.bf16_round
ACTS = {None: lambda x: x, "mish": oracle.mish, "gelu": oracle.gelu_tanh}


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _ulp_close(got, ref, ulps=1.0, frac_exact=0.9, abs_tol=0.0):
    """Stored-bf16 results: every element within `ulps` bf16 ulps of the oracle's rounded value (approximate SFU
    functions and summation order can move a value across a rounding boundary), and most of them identical.
    abs_tol: absolute slack for what is NOT a rounding matter — float32 accumulation noise (a few 1e-6 of the largest
    output, which is many ulps of an output that happens to be ~0) and the absolute error of the approximate activation."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    tol = ulps * bf16_ulp(ref) * (1 + 1e-9) + abs_tol
    bad = np.abs(got - ref) > tol
    assert not bad.any(), f"{bad.sum()} of {bad.size} elements off by more than {ulps} bf16 ulp; worst {np.abs(got - ref).max():.3e}"
    assert (got == ref).mean() >= frac_exact, f"only {(got == ref).mean():.3f} of the elements are bit-identical"


from test_gpu_ops import DENSE_SHAPES  # noqa: E402


@pytest.mark.parametrize("shape", DENSE_SHAPES)
def test_dense_f32_epilogue_against_bf16_operands(shape):
    """The GEMM itself: with operands rounded as the kernel rounds them only float32 accumulation noise is left."""
    from vision_transformer_detector_b200 import ops
    M, K, N = shape
    rng = np.random.default_rng(hash(shape) % 2**31)
    a = rng.normal(size=(M, K)).astype(np.float32)
    w = (rng.normal(size=(K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.normal(size=(N,)).astype(np.float32)
    ref = R(a) @ R(w) + b.astype(np.float64)
    got = ops.dense(_t(a), _t(w), _t(b), mode="bf16").cpu().numpy()
    assert rel_err(got, ref) < 2e-5


@pytest.mark.parametrize("act", ["mish", "gelu", None])
@pytest.mark.parametrize("shape,pair", [((1296, 28, 3584), False), ((1300, 28, 3584), True), ((4096, 3584, 1792), True),
                                        ((640, 3584, 1792), False), ((300, 1792, 896), False), ((2592, 896, 448), True),
                                        ((34, 1296, 8704), False), ((1296, 28, 1536), False), ((130, 200, 300), False),
                                        ((127, 70, 17), False), ((1100, 200, 300), True)])
def test_dense_bf16_store_epilogue(shape, pair, act):
    """The epilogue the product uses between layers: bias + activation on packed float32 pairs (one ex2 + one rcp for
    Mish), bf16 pack, 64B-swizzled staging, TMA store — single-CTA and CTA-pair kernels."""
    from vision_transformer_detector_b200 import ops
    M, K, N = shape
    rng = np.random.default_rng(hash(shape) % 2**31 + 1)
    a = rng.normal(size=(M, K)).astype(np.float32)
    w = (rng.normal(size=(K, N)) * (1.5 / np.sqrt(K))).astype(np.float32)
    b = rng.normal(size=(N,)).astype(np.float32)
    pre = R(a) @ R(w) + b.astype(np.float64)
    ref = R(ACTS[act](pre))
    got = ops.dense_ex(_t(a), _t(w), _t(b), act=act, store_bf16=True, pair=pair).cpu().numpy()
    # float32 accumulation: measured <= 4e-6 of max|pre| (scripts/debug_store_epilogue.py); tanh.approx (GELU) has an
    # absolute error of 2^-11 on tanh, i.e. 2.5e-4 |x| on the output; the fast Mish 4e-7 |x| (test_mish_fast_form_accuracy)
    act_abs = {None: 0.0, "mish": 4e-7, "gelu": 3e-4}[act] * max(1.0, float(np.abs(pre).max()))
    _ulp_close(got, ref, ulps=1.0, frac_exact=0.97 if act != "gelu" else 0.9, abs_tol=1e-5 * float(np.abs(pre).max()) + act_abs)


def test_mish_fast_form_accuracy():
    """x - 2x / (n^2 + 2n + 2) with ex2.approx / rcp.approx, measured in isolation over the whole useful range
    (identity weights, float32 epilogue): absolute error vs the exact Mish, incl. the tails where n overflows."""
    from vision_transformer_detector_b200 import ops
    x = np.concatenate([np.linspace(-30, 30, 128 * 255, dtype=np.float32), [-88.0, -60.0, 60.0, 88.0] * 32]).reshape(-1, 128)
    x = R(x).astype(np.float32)                                 # exactly representable operands: the GEMM is then exact
    eye = np.eye(128, dtype=np.float32)
    got = ops.dense_ex(_t(x), _t(eye), None, act="mish").cpu().numpy()
    ref = oracle.mish(x.astype(np.float64))
    err = np.abs(got - ref)
    # the form subtracts two numbers of size |x|, so its absolute error is a few float32 ulps OF x, whatever the result
    bound = 4e-7 * np.maximum(1.0, np.abs(x.astype(np.float64)))
    assert (err <= bound).all(), float((err / bound).max())
    print("mish fast form: max abs err", float(err.max()), "max err / (4e-7 max(1,|x|))", float((err / bound).max()))


def test_position_add_epilogue():
    """linear_projection + PositionEncoding (det.py:291-307): the per-token scalar is added in the GEMM epilogue."""
    from vision_transformer_detector_b200 import ops
    T, B, K, N = 1296, 2, 867, 28
    rng = np.random.default_rng(5)
    a = rng.uniform(-1, 1, size=(B * T, K)).astype(np.float32)
    w = (rng.normal(size=(K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.normal(size=(N,)).astype(np.float32)
    pos = rng.uniform(-0.05, 0.05, size=(T,)).astype(np.float32)
    ref = R(a) @ R(w) + b.astype(np.float64) + np.tile(pos.astype(np.float64), B)[:, None]
    got = ops.dense_ex(_t(a), _t(w), _t(b), pos=_t(pos)).cpu().numpy()
    assert rel_err(got, ref) < 2e-5


@pytest.mark.parametrize("M,K,N", [(1296 * 2, 320, 28), (1000, 867, 28), (257, 64, 32), (130, 40, 8), (77, 56, 30)])
def test_fused_layernorm_epilogue(M, K, N):
    """attention_output + add + the next LayerNormalization (det.py:364-379) in one epilogue: the float32 residual-stream
    row and its LayerNorm'd bf16 copy, per row."""
    from vision_transformer_detector_b200 import ops
    rng = np.random.default_rng(M + N)
    a = rng.normal(size=(M, K)).astype(np.float32)
    w = (rng.normal(size=(K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.normal(size=(N,)).astype(np.float32)
    r = (rng.normal(size=(M, N)) * 2).astype(np.float32)
    g = rng.uniform(0.5, 1.5, size=(N,)).astype(np.float32)
    be = rng.normal(size=(N,)).astype(np.float32)
    x = R(a) @ R(w) + b.astype(np.float64) + r
    got, ln = ops.dense_ex(_t(a), _t(w), _t(b), resid=_t(r), ln=(_t(g), _t(be), 1e-3))
    got, ln = got.cpu().numpy(), ln.cpu().numpy()
    assert np.abs(got - x).max(axis=1).max() < 2e-5 * np.abs(x).max()              # per-row bound, not a global one
    ln_ref = oracle.layer_norm(got.astype(np.float64), g.astype(np.float64), be.astype(np.float64), 1e-3)
    _ulp_close(ln, R(ln_ref), ulps=1.0, frac_exact=0.97, abs_tol=2e-6 * float(np.abs(ln_ref).max()))    # float32 statistics


@pytest.mark.parametrize("act", ["mish", "gelu"])
@pytest.mark.parametrize("M,widths,with_ln", [(1296 * 3, (224, 112, 56, 28), True), (1000, (224, 112, 56, 28), False),
                                              (130, (64, 32, 16, 8), True), (129, (256, 128, 64, 32), True), (77, (120, 56, 24, 12), True)])
def test_mlp_tail_kernel(M, widths, with_ln, act):
    """The fused last three MLP layers + residual + next LayerNorm (mlp_tail.cu) against the same chain with the
    kernel's roundings: activations between the layers are bf16, the last layer's output stays float32."""
    from vision_transformer_detector_b200 import ops
    K0, N0, N1, N2 = widths
    rng = np.random.default_rng(M + K0)
    a = rng.normal(size=(M, K0)).astype(np.float32)
    ws = [(rng.normal(size=(k, n)) * (1.5 / np.sqrt(k))).astype(np.float32) for k, n in ((K0, N0), (N0, N1), (N1, N2))]
    bs = [rng.normal(size=(n,)).astype(np.float32) * 0.5 for n in (N0, N1, N2)]
    x = rng.normal(size=(M, N2)).astype(np.float32)
    g = rng.uniform(0.5, 1.5, size=(N2,)).astype(np.float32)
    be = rng.normal(size=(N2,)).astype(np.float32)
    f = ACTS[act]
    y = R(f(R(a) @ R(ws[0]) + bs[0].astype(np.float64)))
    y = R(f(y @ R(ws[1]) + bs[1].astype(np.float64)))
    ref = f(y @ R(ws[2]) + bs[2].astype(np.float64)) + x
    layers = [(_t(w), _t(b)) for w, b in zip(ws, bs)]
    if with_ln:
        got, ln = ops.mlp_tail(_t(a), layers, _t(x), act=act, ln=(_t(g), _t(be), 1e-3))
        ln = ln.cpu().numpy()
    else:
        got = ops.mlp_tail(_t(a), layers, _t(x), act=act)
    got = got.cpu().numpy()
    # one-ulp flips of the intermediate bf16 activations reach the output scaled by one weight: ~1e-3 of the row
    assert np.abs(got - ref).max() < 3e-3 * np.abs(ref).max()
    assert np.sqrt(np.mean((got - ref) ** 2)) < 2e-4 * np.abs(ref).max()
    if with_ln:
        ln_ref = oracle.layer_norm(got.astype(np.float64), g.astype(np.float64), be.astype(np.float64), 1e-3)
        _ulp_close(ln, R(ln_ref), ulps=1.0, frac_exact=0.97, abs_tol=2e-6 * float(np.abs(ln_ref).max()))


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("B,T,D,S", [(2, 1296, 28, 17), (3, 36, 28, 17), (2, 25, 28, 17), (1, 1600, 768, 17), (2, 7, 12, 5),
                                     (2, 101, 768, 17), (1, 50, 64, 32), (3, 333, 132, 17)])
def test_head_slots_kernel(B, T, D, S, mode):
    """Dense(D -> 17) per token + Reshape((17, -1)) (det.py:454-463): the flat reinterpretation, incl. token counts that
    are not a multiple of the 16-byte row pitch (rows padded in memory, invisible at the boundary)."""
    from vision_transformer_detector_b200 import ops
    rng = np.random.default_rng(T + D)
    x = rng.normal(size=(B, T, D)).astype(np.float32)
    w = (rng.normal(size=(D, S)) / np.sqrt(D)).astype(np.float32)
    b = rng.normal(size=(S,)).astype(np.float32)
    ref = (x.astype(np.float64) @ w.astype(np.float64) + b).reshape(B, S, T)          # det.py:461: same memory, new shape
    got = ops.head_slots(_t(x), _t(w), _t(b), mode=mode).cpu().numpy()
    assert got.shape == (B, S, T)
    if mode == "fp32":
        assert rel_err(got, ref) < 1e-6
    else:
        _ulp_close(got, R(ref), ulps=1.0, frac_exact=0.98, abs_tol=2e-6 * float(np.abs(ref).max()))    # float32 dot product of D terms


@pytest.mark.parametrize("B,T,H,d", [(2, 1296, 8, 40), (1, 4096, 2, 40), (2, 1600, 3, 64), (3, 100, 2, 40), (1, 64, 1, 8), (2, 65, 2, 24),
                                     (5, 129, 3, 40), (2, 300, 1, 16)])
def test_attention_kernels_against_bf16_operands(B, T, H, d):
    """The attention kernel with q, k, v already bf16 and the probabilities rounded to bf16 in the oracle as in the kernel;
    image-boundary cases (T = 65, 129, 300) put keys and queries of the NEXT image into the last tiles, which the masks must
    keep out."""
    from vision_transformer_detector_b200 import ops
    rng = np.random.default_rng(B * T + d)
    q, k, v = (R(rng.normal(size=(B, T, H, d)) * 1.5) for _ in range(3))
    ref = R(oracle.attention_core_bf16(q, k, v))
    got = ops.attention(_t(q), _t(k), _t(v), mode="bf16").cpu().numpy()
    err = np.abs(got - ref)
    # the stored context is bf16 (one ulp of slack per element); P is rounded against a different reference point
    assert (err <= bf16_ulp(ref) + 2e-3 * np.abs(ref).max()).all(), float((err / np.abs(ref).max()).max())
    assert np.sqrt(np.mean(err ** 2)) < 8e-4 * np.abs(ref).max()


@pytest.mark.parametrize("B,T,H,d", [(2, 300, 3, 96), (1, 1296, 2, 128), (2, 65, 2, 72), (1, 129, 5, 104), (1, 1600, 2, 80)])
def test_attention_wide_heads_against_bf16_operands(B, T, H, d):
    """Heads wider than 64 (the reference accepts any key_dim): the kernel's two-box form — Q / K / V tiles of two 64-column
    boxes, QK^T over up to eight k-steps, PV as two 64-column products, O in 128 TMEM columns, one CTA per SM."""
    from vision_transformer_detector_b200 import ops
    rng = np.random.default_rng(B * T + d)
    q, k, v = (R(rng.normal(size=(B, T, H, d)) * 1.5) for _ in range(3))
    ref = R(oracle.attention_core_bf16(q, k, v))
    got = ops.attention(_t(q), _t(k), _t(v), mode="bf16").cpu().numpy()
    err = np.abs(got - ref)
    assert (err <= bf16_ulp(ref) + 2e-3 * np.abs(ref).max()).all(), float((err / np.abs(ref).max()).max())
    assert np.sqrt(np.mean(err ** 2)) < 8e-4 * np.abs(ref).max()


# ------------------------------------------------------------------------------------------------
# whole model
# ------------------------------------------------------------------------------------------------
MEASURED = {}


def _bf16_tensor_close(got, ref, ulps=6.0, frac_within_one=0.85):
    """A stored bf16 activation at the end of a chain of bf16-stored layers (head_last: seven of them after the encoder):
    one-ulp rounding flips upstream reach an element through hundreds of weights, so individual elements move by a few
    units u = bf16 ulp + 1e-3 max|ref| (measured on the default model: worst 4.0 u, 89 % within one)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    e = np.abs(got - ref)
    u = bf16_ulp(ref) + 1e-3 * np.abs(ref).max()
    assert (e <= ulps * u).all(), float((e / u).max())
    assert (e <= u).mean() >= frac_within_one, float((e <= u).mean())


def _taps(m, batch, L):
    return {n: m.debug_read(n, batch) for n in ["embedded_patches"] + [f"block_{i + 1}" for i in range(L)] + ["head_last"]}


@pytest.mark.parametrize("cfg_kw,batch", [({}, 5), (dict(use_mish=False), 3),
                                          (dict(input_shape=(100, 100, 3)), 3),                    # 36 tokens: not a multiple of 8
                                          (dict(input_shape=(70, 70, 3)), 2),                      # 25 tokens: odd
                                          (dict(input_shape=(64, 64, 3), patch_size=16, embedding_dim=64, encoder_num_heads=4,
                                                encoder_key_dim=64, encoder_mlp_quantities=3), 2)])
def test_tiny_models_against_the_bf16_faithful_oracle(cfg_kw, batch):
    cfg = tiny_config(**cfg_kw)
    w = vd.random_weights(cfg, seed=11, spread=True)
    x = images(cfg, batch)
    ref, inter = oracle.forward_bf16(w, cfg, x, return_intermediates=True)
    m = build_model(cfg, w, "bf16")
    m.debug_taps(True)
    got = m.predict(x)
    taps = _taps(m, batch, cfg.encoder_repeat_times)
    for name in ("embedded_patches", "block_1", "block_2"):
        assert rel_err(taps[name], inter[name]) < 2e-3, name
    # head_last is a STORED bf16 tensor: a flip of the last bit of its largest element alone is 4e-3..8e-3 of max|ref|
    _bf16_tensor_close(taps["head_last"], inter["head_last"])
    assert rel_err(got, ref) < 1e-2
    # the float32 mode accepts the same ragged token counts
    m32 = build_model(cfg, w, "fp32")
    assert rel_err(m32.predict(x), oracle.forward(w, cfg, x, np.float64)) < 1e-3
    m.close(); m32.close()


def test_default_model_against_the_bf16_faithful_oracle_per_block():
    cfg = vd.DetectorConfig()
    w = vd.random_weights(cfg, seed=1, spread=True)
    x = images(cfg, 1)
    ref, inter = oracle.forward_bf16(w, cfg, x, return_intermediates=True)
    m = build_model(cfg, w, "bf16")
    m.debug_taps(True)
    got = m.predict(x)
    taps = _taps(m, 1, cfg.encoder_repeat_times)
    errs = {n: rel_err(taps[n], inter[n]) for n in taps}
    errs["logits"] = rel_err(got, ref)
    print("bf16 kernels vs bf16-faithful oracle, default model:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["embedded_patches"] < 1e-4
    assert max(errs[f"block_{i + 1}"] for i in range(8)) < 1e-3           # measured 1.7e-4 (block 1) ... 4.4e-4 (block 8)
    _bf16_tensor_close(taps["head_last"], inter["head_last"])
    # seven bf16-stored head layers after the encoder: flips accumulate; measured 7e-3, the same size as the distance
    # of either side to the float64 reference
    assert errs["logits"] < 1.5e-2
    m.close()


@pytest.mark.parametrize("option,value", [("fuse_ln", 0), ("fuse_tail", 0), ("gemm_pair", 0), ("gemm_pair", 2)])
def test_fused_and_unfused_builds_agree(option, value):
    """Every fusion / kernel-selection switch must leave the result unchanged up to bf16 rounding: the stand-alone
    LayerNorm kernel vs the GEMM epilogue, three GEMM launches vs the fused MLP tail, single-CTA vs CTA-pair GEMM — per
    encoder block (taps) and on the logits."""
    cfg = vd.DetectorConfig()
    w = vd.random_weights(cfg, seed=1, spread=True)
    x = images(cfg, 2)
    m = build_model(cfg, w, "bf16")
    m.debug_taps(True)
    base = m.predict(x)
    base_taps = _taps(m, 2, 8)
    m.set_option(option, value)
    assert m.get_option(option) == value
    alt = m.predict(x)
    alt_taps = _taps(m, 2, 8)
    for n in base_taps:
        if n == "head_last":
            _bf16_tensor_close(alt_taps[n], base_taps[n])
        else:
            e = rel_err(alt_taps[n], base_taps[n])
            assert e < 1e-3, (n, e)
    assert rel_err(alt, base) < 1.5e-2
    m.close()


@pytest.mark.parametrize("cfg_kw,batch", [(dict(), 3), (dict(input_shape=(60, 130, 3), encoder_num_heads=2, encoder_mlp_quantities=3,
                                                             encoder_repeat_times=2, mlp_head_last_units=8, mlp_head_dense_layers_quantity=2), 6)])
def test_changing_one_image_leaves_the_others_bit_identical(cfg_kw, batch):
    """Images are independent: cross-image leakage (a key tile that straddles two images, a row tile shared by two
    images' tokens) would show up as a changed neighbour.  Default config: 1296 tokens = 10 full key tiles + 16 keys."""
    cfg = vd.DetectorConfig(**cfg_kw)
    w = vd.random_weights(cfg, seed=1, spread=True)
    x = images(cfg, batch)
    m = build_model(cfg, w, "bf16")
    base = m.predict(x)
    for victim in (0, batch - 1, batch // 2):
        y = x.copy()
        y[victim] = -y[victim][::-1]
        out = m.predict(y)
        others = [i for i in range(batch) if i != victim]
        assert np.array_equal(out[others], base[others])
        assert not np.array_equal(out[victim], base[victim])
    m.close()
