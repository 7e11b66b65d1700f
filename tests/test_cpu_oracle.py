"""CPU suite (-m "not gpu"): pins the oracle restatement to what the reference's own code returned (its naive test
oracles, shape rules, BN fold, quantisation helpers and x86 INT8 convolution, compiled into oracle/_ref by
`make -C oracle ref`; their results are stored in tests/golden/reference_oracle.json) and to the committed golden
fixtures; property tests of the oracle itself."""
import hashlib
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# What the reference returned for every case below, so that the comparison runs without the reference's sources: a
# SHA-256 digest per output array (the arrays themselves come to megabytes) and plain JSON for scalars and shapes.
# `B200_RECORD_REFERENCE=1 pytest tests/test_cpu_oracle.py`, with oracle/_ref built, re-runs the reference on the same
# seeded inputs and rewrites the stored results.
REF_GOLD = os.path.join(GOLD, "reference_oracle.json")


def _digest(a):
    """dtype, shape and SHA-256 of an array; -0.0 counts as 0.0 and all NaNs as one, as in assert_array_equal."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a).astype(a.dtype) + a.dtype.type(0)
    return "%s%s %s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest())


class _Reference:
    def __init__(self, stored, record):
        self.stored, self.record, self.new = stored, record, {}

    def value(self, key, run):
        """The reference's result for case `key`: run() when recording, the stored result otherwise."""
        if self.record:
            self.new[key] = json.loads(json.dumps(run()))
            return self.new[key]
        assert key in self.stored, "no stored reference result for %r (re-record %s)" % (key, REF_GOLD)
        return self.stored[key]

    def assert_equal(self, key, got, run):
        """`got` is bit for bit the array the reference returned for case `key` (run() when recording)."""
        assert _digest(got) == self.value(key, lambda: _digest(run())), "differs from the reference: %r" % key


@pytest.fixture(scope="module")
def reference(oracle):
    record = os.environ.get("B200_RECORD_REFERENCE") == "1"
    if record and oracle.ref_lib() is None:
        raise RuntimeError("B200_RECORD_REFERENCE=1 needs oracle/_ref (make -C oracle ref)")
    with open(REF_GOLD) as f:
        stored = json.load(f)
    ref = _Reference(stored, record)
    yield ref
    if record:
        stored.update(ref.new)
        with open(REF_GOLD, "w") as f:       # one case per line
            f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(v)) for k, v in sorted(stored.items())))


# shape sweep of reference test/saber/test_saber_conv.cpp:886-901,1000-1015
@pytest.mark.parametrize("k,pad,stride,dil", [(1, 0, 1, 1), (3, 1, 1, 1), (3, 1, 2, 1), (3, 0, 1, 2), (3, 1, 2, 2)])
@pytest.mark.parametrize("cin,cout,hw,n", [(4, 4, 12, 1), (8, 32, 21, 3), (16, 8, 24, 1)])
@pytest.mark.parametrize("bias,relu", [(True, True), (False, False)])
def test_conv_f32_matches_reference_oracle(oracle, reference, k, pad, stride, dil, cin, cout, hw, n, bias, relu):
    rng = np.random.default_rng(k * 100 + cin)
    x = rng.uniform(-5, 5, (n, cin, hw, hw)).astype(np.float32)
    w = rng.uniform(-1, 1, (cout, cin, k, k)).astype(np.float32)
    b = rng.uniform(-1, 1, cout).astype(np.float32) if bias else None
    kw = dict(stride=(stride, stride), pad=(pad, pad), dil=(dil, dil), relu=relu)
    a = oracle.conv_f32_nchw(x, w, b, **kw)
    reference.assert_equal("conv_f32%r" % ((k, pad, stride, dil, cin, cout, hw, n, bias, relu),), a,
                           lambda: oracle.ref_conv_f32_nchw(x, w, b, **kw))
    # the vectorised NHWC variant only re-associates the dot product
    fast = oracle.conv_f32_nhwc(np.transpose(x, (0, 2, 3, 1)), w, b, **kw)
    mr, md = oracle.tensor_cmp(np.transpose(a, (0, 2, 3, 1)), fast)
    assert md <= 1e-5 * max(1.0, float(np.abs(a).max())), (mr, md)


def test_conv_f32_real_model_shape(oracle, reference):
    """test_saber_conv.cpp:868-883: 1x3x224x224 -> 64, 3x3, pad 1, bias + relu."""
    rng = np.random.default_rng(0)
    x = rng.uniform(-5, 5, (1, 3, 224, 224)).astype(np.float32)
    w = rng.uniform(-1, 1, (64, 3, 3, 3)).astype(np.float32)
    b = rng.uniform(-1, 1, 64).astype(np.float32)
    reference.assert_equal("conv_f32 1x3x224x224 -> 64", oracle.conv_f32_nchw(x, w, b, pad=(1, 1), relu=True),
                           lambda: oracle.ref_conv_f32_nchw(x, w, b, pad=(1, 1), relu=True))


def test_conv_f32_groups_beta_alpha(oracle, reference):
    rng = np.random.default_rng(1)
    x = rng.uniform(-2, 2, (2, 8, 9, 9)).astype(np.float32)
    w = rng.uniform(-1, 1, (8, 2, 3, 3)).astype(np.float32)
    dst = rng.uniform(-1, 1, (2, 8, 9, 9)).astype(np.float32)
    kw = dict(group=4, pad=(1, 1), beta=0.5, alpha=1.5, dst=dst)
    reference.assert_equal("conv_f32 groups beta alpha", oracle.conv_f32_nchw(x, w, None, **kw),
                           lambda: oracle.ref_conv_f32_nchw(x, w, None, **kw))


@pytest.mark.parametrize("unsigned", [False, True])
@pytest.mark.parametrize("k,pad,stride", [(1, 0, 1), (3, 1, 1), (3, 1, 2)])
@pytest.mark.parametrize("elt,relu,down", [(False, True, False), (True, True, False), (True, False, True)])
def test_conv_int8_basic_matches_reference_oracle(oracle, reference, unsigned, k, pad, stride, elt, relu, down):
    rng = np.random.default_rng(7 + k + stride)
    x = (rng.integers(0, 256, (2, 10, 10, 8)).astype(np.uint8) if unsigned
         else rng.integers(-128, 128, (2, 10, 10, 8)).astype(np.int8))
    w = rng.integers(-127, 128, (16, 8, k, k)).astype(np.int8)
    b = rng.integers(-500, 500, 16).astype(np.int32)
    sc = rng.uniform(0.001, 0.01, 16).astype(np.float32)
    oh = oracle.conv_out_size(10, pad, 1, k, stride)
    dst = rng.integers(-128, 128, (2, oh, oh, 16)).astype(np.int8)
    kw = dict(pad=(pad, pad), stride=(stride, stride), relu=relu, has_elt_sum=elt, sum_scale=0.7, dst=dst,
              round_down=down)
    a = oracle.conv_s8_nhwc_basic(x, w, b, sc, **kw)
    reference.assert_equal("conv_int8_basic%r" % ((unsigned, k, pad, stride, elt, relu, down),), a,
                           lambda: oracle.conv_s8_nhwc_basic(x, w, b, sc, use_ref=True, **kw))


def test_x86_semantics_agree_with_reference_oracle_on_shared_subset(oracle, reference):
    """The x86-JIT restatement and conv_basic_check_int8 coincide when the bias is integral, the
    output is s8 and there is no residual -- pins oracle_conv_s8_nhwc_x86 to the reference."""
    rng = np.random.default_rng(11)
    x = rng.integers(-128, 128, (2, 9, 9, 16)).astype(np.int8)
    w = rng.integers(-127, 128, (32, 16, 3, 3)).astype(np.int8)
    b = rng.integers(-1000, 1000, 32).astype(np.int32)
    sc = rng.uniform(0.0005, 0.005, 32).astype(np.float32)
    for relu in (False, True):
        j = oracle.conv_s8_nhwc_x86(x, w, b.astype(np.float32), sc, pad=(1, 1), relu=relu, out_dtype=oracle.DT_INT8)
        reference.assert_equal("conv_int8_basic shared subset relu=%r" % relu, j,
                               lambda: oracle.conv_s8_nhwc_basic(x, w, b, sc, pad=(1, 1), relu=relu, use_ref=True))


@pytest.mark.parametrize("ptype", [1, 2, 3])
@pytest.mark.parametrize("unsigned", [False, True])
def test_pool_int8_matches_reference_oracle(oracle, reference, ptype, unsigned):
    rng = np.random.default_rng(3)
    x = (rng.integers(0, 128, (2, 13, 13, 8)).astype(np.uint8) if unsigned
         else rng.integers(0, 128, (2, 13, 13, 8)).astype(np.int8))
    a = oracle.pool_s8_nhwc(x, (3, 3), (1, 1), (2, 2), ptype)
    reference.assert_equal("pool_int8%r" % ((ptype, unsigned),), a,
                           lambda: oracle.pool_s8_nhwc(x, (3, 3), (1, 1), (2, 2), ptype, use_ref=True))


def test_tensor_cmp_matches_reference(oracle, reference):
    rng = np.random.default_rng(5)
    a = rng.uniform(-3, 3, 1000).astype(np.float32)
    b = a + rng.uniform(-1e-3, 1e-3, 1000).astype(np.float32)
    want = reference.value("tensor_cmp", lambda: oracle.tensor_cmp(a, b, use_ref=True))
    assert oracle.tensor_cmp(a, b) == pytest.approx(tuple(want), rel=1e-12)


def test_pool_shape_rule(oracle):
    # Caffe ceil mode with the pad clamp (saber/funcs/pooling.h:96-125)
    assert oracle.pool_out_size(112, 112, 3, 3, 0, 0, 2, 2) == (56, 56)
    assert oracle.pool_out_size(224, 224, 2, 2, 0, 0, 2, 2) == (112, 112)
    assert oracle.pool_out_size(7, 7, 3, 3, 1, 1, 2, 2) == (4, 4)
    assert oracle.pool_out_size(6, 6, 3, 3, 1, 1, 2, 2) == (4, 4)
    assert oracle.pool_out_size(5, 5, 2, 2, 1, 1, 2, 2) == (3, 3)      # ceil gives 4, the clamp drops one
    assert oracle.pool_out_size(13, 13, 3, 3, 0, 0, 2, 2, floor_as_conv=True) == (6, 6)
    assert oracle.pool_out_size(7, 7, 7, 7, 0, 0, 1, 1, global_pooling=True) == (1, 1)


def test_pool_shape_rule_matches_reference_compute_output_shape(oracle, reference):
    """Exhaustive sweep of the restated rule -- and of the product's host-side b200_pool_out_hw -- against the
    reference's own Pooling::compute_output_shape compiled from saber/funcs/pooling.h (oracle/_ref)."""
    import ctypes as C
    from anakin_b200 import saber_abi as A
    lib = A.load()
    sizes = [(7, 7), (12, 13), (14, 14), (21, 24), (56, 56), (112, 112), (224, 224)]
    cases = [(h, w, win, pad, stride, floor) for h, w in sizes for win in (1, 2, 3, 5, 7) for pad in (0, 1, 2, 3)
             for stride in (1, 2, 3) for floor in (False, True) if not (win > h + 2 * pad or pad >= win)]
    wants = reference.value("pool_out_size sweep", lambda: [
        oracle.ref_pool_out_size(h, w, win, win, pad, pad, stride, stride, False, floor)
        for h, w, win, pad, stride, floor in cases])
    assert len(wants) == len(cases) > 500
    for (h, w, win, pad, stride, floor), want in zip(cases, wants):
        want = tuple(want)
        assert oracle.pool_out_size(h, w, win, win, pad, pad, stride, stride, False, floor) == want, \
            (h, w, win, pad, stride, floor)
        d = A.PoolDesc()
        d.dtype, d.type, d.n, d.h, d.w, d.c = A.FLOAT, 1, 1, h, w, 16
        d.window_h = d.window_w = win
        d.pad_h = d.pad_w = pad
        d.stride_h = d.stride_w = stride
        d.global_pooling, d.floor_as_conv = 0, int(floor)
        oh, ow = C.c_int32(), C.c_int32()
        assert lib.b200_pool_out_hw(C.byref(d), C.byref(oh), C.byref(ow)) == A.SUCCESS
        assert (oh.value, ow.value) == want, (h, w, win, pad, stride, floor)
    wants = reference.value("pool_out_size global sweep", lambda: [
        oracle.ref_pool_out_size(h, w, 3, 3, 0, 0, 1, 1, True) for h, w in sizes])
    for (h, w), want in zip(sizes, wants):
        assert oracle.pool_out_size(h, w, 3, 3, 0, 0, 1, 1, True) == tuple(want)


@pytest.mark.parametrize("conv_bias", [False, True])
@pytest.mark.parametrize("scale_bias", [False, True])
@pytest.mark.parametrize("factor", [1.0, 0.0, 0.999])
def test_bn_fold_matches_reference_update_weights(oracle, reference, conv_bias, scale_bias, factor):
    """oracle_fold_bn_scale vs the reference's WeightsFusion<float,X86>::update_weights compiled from
    framework/utils/parameter_fusion.cpp:86-131 (oracle/_ref): bit-exact folded weights and bias."""
    rng = np.random.default_rng(int(conv_bias) * 4 + int(scale_bias) * 2 + int(factor * 10))
    k, c, r = 37, 19, 3
    w = rng.standard_normal((k, c, r, r)).astype(np.float32)
    b = rng.uniform(-1, 1, k).astype(np.float32) if conv_bias else None
    mean = rng.uniform(-0.1, 0.1, k).astype(np.float32)
    var = rng.uniform(0.5, 1.5, k).astype(np.float32)
    gamma = rng.uniform(0.8, 1.2, k).astype(np.float32)
    beta = rng.uniform(-0.1, 0.1, k).astype(np.float32) if scale_bias else None
    got = oracle.fold_bn_scale(w, b, factor, 1e-5, mean, var, gamma, beta)
    for i, what in enumerate(("weights", "bias")):
        reference.assert_equal("bn_fold %s%r" % (what, (conv_bias, scale_bias, factor)), got[i],
                               lambda: oracle.ref_fold_bn_scale(w, b, factor, 1e-5, mean, var, gamma, beta)[i])


# (input unsigned, output dtype, relu): the dtype pairs GemmX8S8S32XConv::dispatch accepts (gemm_x8s8s32x_conv.cpp:287-306);
# u8 output only with relu -- without it the reference casts negative values with wrap-around (no saturation)
_GEMM_CONV_DTYPES = [(True, 7, True), (True, 1, False), (True, 1, True), (False, 3, False), (False, 3, True),
                     (False, 7, True), (False, 1, False)]


@pytest.mark.parametrize("xu,odt,relu", _GEMM_CONV_DTYPES)
@pytest.mark.parametrize("k,pad,stride,dil", [(1, 0, 1, 1), (3, 1, 1, 1), (3, 1, 2, 1), (3, 0, 1, 1), (1, 0, 2, 1), (3, 2, 1, 2)])
def test_x86_int8_conv_matches_reference_gemm_conv(oracle, reference, xu, odt, relu, k, pad, stride, dil):
    """The INT8 pipeline the CUDA path is held to -- per-channel weight quantisation, bias pre-scaling, the
    input/output dtype scale table, integer accumulation, (acc + bias) * scale, relu, round-to-nearest-even -- against
    the reference's own x86 INT8 convolution GemmX8S8S32XConv run verbatim (oracle/_ref; only MKL's integer GEMM is a
    stand-in): bit-exact for every dtype pair it supports, bias on and off."""
    rng = np.random.default_rng(hash((xu, odt, relu, k, pad, stride, dil)) % 2 ** 31)
    for (n, hw, cin, cout), with_bias in [((1, 12, 16, 32), True), ((3, 21, 8, 4), False), ((2, 7, 64, 40), True)]:
        x = rng.integers(0, 256, (n, hw, hw, cin)).astype(np.uint8) if xu else rng.integers(-128, 128, (n, hw, hw, cin)).astype(np.int8)
        w = (rng.standard_normal((cout, cin, k, k)) * rng.uniform(0.02, 0.3, (cout, 1, 1, 1))).astype(np.float32)
        bias = rng.uniform(-0.5, 0.5, cout).astype(np.float32) if with_bias else None
        in_scale = 0.0173
        kw = dict(stride=(stride, stride), pad=(pad, pad), dil=(dil, dil))
        case = "gemm_conv%r" % ((xu, odt, relu, k, pad, stride, dil, n, hw, cin, cout, with_bias),)
        # an output scale under which nothing leaves the 8-bit range (the reference's cast does not saturate)
        out_scale = reference.value(case + " out_scale", lambda: float(np.abs(
            oracle.ref_gemm_conv_int8(x, w, bias, in_scale, 1, 1.0, relu=relu, **kw)).max()) / 120.0 + 1e-6)
        wq, ws = oracle.quant_weights_per_oc(w)
        sc, bf, _ = oracle.int8_conv_scales(ws, bias, in_scale, 7 if xu else 3, out_scale, odt)
        got = oracle.conv_s8_nhwc_x86(x, wq, bf if with_bias else None, sc, out_dtype=odt, relu=relu, **kw)
        reference.assert_equal(case, got, lambda: oracle.ref_gemm_conv_int8(x, w, bias, in_scale, odt, out_scale,
                                                                             relu=relu, **kw))


def test_int8_quantisation_helpers_match_reference_scale_utils(oracle, reference):
    """The x86 INT8 quantisation rules restated in oracle.c vs the reference's own utils::ScaleUtils
    (saber/funcs/impl/x86/x86_utils.h:293-372) compiled into oracle/_ref: per-output-channel weight quantisation
    (truncating cast), activation quantisation to s8 (roundf + clamp) and to u8 (scale * 127/255, truncation)."""
    rng = np.random.default_rng(11)
    w = (rng.standard_normal((48, 20, 3, 3)) * rng.uniform(0.01, 3.0, (48, 1, 1, 1))).astype(np.float32)
    got = oracle.quant_weights_per_oc(w)
    for i, what in enumerate(("weights", "scales")):
        reference.assert_equal("quant_weights_per_oc " + what, got[i], lambda: oracle.ref_quant_weights_per_oc(w)[i])
    x = np.concatenate([rng.uniform(-3, 3, 5000), [0.5, -0.5, 1.5, -1.5, 2.5, 126.5, 127.5, -128.5, 3e4, -3e4]]).astype(np.float32)
    for scale in (0.013, 0.02362, 1.0):
        reference.assert_equal("quant_fp32_s8 scale=%r" % scale, oracle.quant_fp32_s8(x * scale, scale),
                               lambda: oracle.ref_quant_fp32(x * scale, scale))
    xu = np.concatenate([rng.uniform(0, 3, 5000), [0.0, 0.999, 1.0, 254.9, 255.0]]).astype(np.float32)
    for scale in (0.013, 0.02362):
        reference.assert_equal("quant_fp32_u8 scale=%r" % scale, oracle.quant_fp32_u8(xu * scale * 127 / 255, scale),
                               lambda: oracle.ref_quant_fp32(xu * scale * 127 / 255, scale, unsigned=True))


def test_bn_fold_equals_unfused_ops(oracle):
    """parameter_fusion.cpp:86-131: conv -> BN -> Scale equals the folded conv."""
    rng = np.random.default_rng(9)
    x = rng.uniform(-1, 1, (1, 6, 6, 4)).astype(np.float32)
    w = rng.uniform(-1, 1, (8, 4, 3, 3)).astype(np.float32)
    b = rng.uniform(-1, 1, 8).astype(np.float32)
    mean, var = rng.uniform(-0.2, 0.2, 8).astype(np.float32), rng.uniform(0.5, 1.5, 8).astype(np.float32)
    gamma, beta = rng.uniform(0.5, 1.5, 8).astype(np.float32), rng.uniform(-0.3, 0.3, 8).astype(np.float32)
    wf, bf = oracle.fold_bn_scale(w, b, 2.0, 1e-5, mean, var, gamma, beta)
    fused = oracle.conv_f32_nhwc(x, wf, bf, pad=(1, 1))
    y = oracle.conv_f32_nhwc(x, w, b, pad=(1, 1))
    y = (y - mean / 2.0) / np.sqrt(var / 2.0 + 1e-5) * gamma + beta
    np.testing.assert_allclose(fused, y, rtol=2e-5, atol=2e-5)


def test_int8_conv_linearity_property(oracle):
    """Size-independent property: with fp32 output and unit scale the x86 int8 conv is exactly
    linear in its input (s32 accumulation is exact)."""
    rng = np.random.default_rng(13)
    a = rng.integers(-60, 60, (1, 14, 14, 32)).astype(np.int8)
    b = rng.integers(-60, 60, (1, 14, 14, 32)).astype(np.int8)
    w = rng.integers(-127, 128, (16, 32, 3, 3)).astype(np.int8)
    f = lambda t: oracle.conv_s8_nhwc_x86(t, w, None, None, pad=(1, 1), out_dtype=oracle.DT_FLOAT)
    np.testing.assert_array_equal(f(a) + f(b), f((a.astype(np.int16) + b).astype(np.int8)))


def test_quantisation_rules(oracle):
    x = np.array([0.0, 0.49, 0.5, 1.5, -0.5, -1.5, 200.0, -200.0], np.float32)
    # secur_cast2char: roundf (half away from zero) then clamp (x86_utils.h:318-324)
    np.testing.assert_array_equal(oracle.quant_fp32_s8(x, 1.0), np.array([0, 0, 1, 2, -1, -2, 127, -128], np.int8))
    # weights: truncating static_cast<char>(w / (max|w|/127)) (x86_utils.h:293-323)
    q, s = oracle.quant_weights_per_oc(np.array([[1.0, -0.999, 0.5, 0.004]], np.float32))
    assert s[0] == np.float32(1.0 / 127.0)
    np.testing.assert_array_equal(q, np.array([[127, -126, 63, 0]], np.int8))


@pytest.mark.parametrize("model", ["tiny_resnet", "tiny_mobilenet", "resnet50", "mobilenet_v1"])
def test_model_walker_reproduces_golden(model, oracle):
    """The committed golden outputs are what the oracle produces today (guards oracle drift)."""
    from anakin_b200 import modelzoo
    from oracle import model_walker as W
    gold = np.load(os.path.join(GOLD, "%s_golden.npz" % model))
    hw = 32 if model.startswith("tiny") else 224
    n = 2
    g = modelzoo.build(model, batch=1)
    x = modelzoo.synthetic_input(n, hw)
    np.testing.assert_array_equal(W.run_fp32(g, x)["prob_out"], gold["prob_fp32"][:n])
    scales = {k: float(np.float32(v)) for k, v in modelzoo.load_calibration(model).items()}
    got = W.run_int8(g, x, scales)["prob_out"]
    np.testing.assert_array_equal(got, gold["prob_int8"][:n])
    assert (got.argmax(1) == gold["top1_int8"][:n]).all()


@pytest.mark.parametrize("model", ["tiny_resnet", "tiny_mobilenet", "resnet50"])
def test_baseline_arm_walker_equals_the_scalar_walker(model, oracle):
    """bench.py's CPU arm (run_int8(fast=True, weight_cache=...): VNNI convolutions with cached weight packs, AVX-512
    pooling) gives the golden outputs, on the first call (cache being filled) and on a second one (cache reused)."""
    from anakin_b200 import modelzoo
    from oracle import model_walker as W
    gold = np.load(os.path.join(GOLD, "%s_golden.npz" % model))
    n = 2
    g = modelzoo.build(model, batch=1)
    x = modelzoo.synthetic_input(n, 32 if model.startswith("tiny") else 224)
    scales = {k: float(np.float32(v)) for k, v in modelzoo.load_calibration(model).items()}
    cache = {}
    for _ in range(2):
        got = W.run_int8(g, x, scales, fast=True, weight_cache=cache)["prob_out"]
        np.testing.assert_array_equal(got, gold["prob_int8"][:n])
    assert cache


def test_softmax_eltwise_activation_oracles(oracle):
    rng = np.random.default_rng(2)
    x = rng.uniform(-5, 5, (4, 10)).astype(np.float32)
    p = oracle.softmax_f32(x, 4, 10, 1)
    e = np.exp(x - x.max(1, keepdims=True))
    np.testing.assert_allclose(p, e / e.sum(1, keepdims=True), rtol=1e-6)
    a, b = rng.uniform(-1, 1, 50).astype(np.float32), rng.uniform(-1, 1, 50).astype(np.float32)
    np.testing.assert_array_equal(oracle.eltwise_f32(a, b, 2, 1.0, 1.0, True), np.maximum(a + b, 0))
    np.testing.assert_array_equal(oracle.activation_f32(a, 2, 0.0), np.maximum(a, 0))


# ---- the restated op oracles against the reference's own test oracles (test_saber_{pooling,fc,softmax,eltwise,
# activation}.cpp function templates, compiled from /root/reference into oracle/_ref by `make -C oracle ref`)
@pytest.mark.parametrize("ptype", [1, 2, 3])            # max, avg incl. padding, avg excl. padding
@pytest.mark.parametrize("window,pad,stride", [((2, 2), (0, 0), (2, 2)), ((3, 3), (1, 1), (2, 2)), ((3, 3), (0, 0), (2, 2)),
                                               ((3, 2), (1, 0), (1, 2)), ((2, 2), (1, 1), (1, 1)), ((7, 7), (0, 0), (1, 1))])
def test_pool_f32_matches_reference_test_oracle(oracle, reference, ptype, window, pad, stride):
    rng = np.random.default_rng(hash((ptype, window, pad, stride)) % 2 ** 31)
    for shape in [(1, 3, 7, 7), (2, 4, 12, 21), (3, 2, 24, 24)]:
        x = rng.uniform(-1, 1, shape).astype(np.float32)
        reference.assert_equal("pool_f32%r" % ((ptype, window, pad, stride, shape),),
                               oracle.pool_f32(x, window, pad, stride, ptype),
                               lambda: oracle.ref_pool_f32(x, window, pad, stride, ptype))


@pytest.mark.parametrize("m,k,n", [(1, 16, 4), (3, 100, 37), (8, 2048, 1000), (2, 25088, 16)])
@pytest.mark.parametrize("bias", [False, True])
def test_fc_f32_matches_reference_test_oracle(oracle, reference, m, k, n, bias):
    rng = np.random.default_rng(m * 131 + k + n)
    x = rng.uniform(-1, 1, (m, k)).astype(np.float32)
    w = rng.uniform(-1, 1, (n, k)).astype(np.float32)
    b = rng.uniform(-1, 1, n).astype(np.float32) if bias else None
    reference.assert_equal("fc_f32%r" % ((m, k, n, bias),), oracle.fc_f32(x, w, b), lambda: oracle.ref_fc_f32(x, w, b))


@pytest.mark.parametrize("shape", [(1, 1000, 1, 1), (8, 1000, 1, 1), (2, 5, 3, 4), (3, 21, 7, 2)])
@pytest.mark.parametrize("axis", [1, 2, 3])
def test_softmax_matches_reference_test_oracle(oracle, reference, shape, axis):
    rng = np.random.default_rng(sum(shape) + axis)
    x = rng.uniform(-6, 6, shape).astype(np.float32)
    outer, inner = int(np.prod(shape[:axis])), int(np.prod(shape[axis + 1:]))
    reference.assert_equal("softmax%r" % ((shape, axis),), oracle.softmax_f32(x, outer, shape[axis], inner),
                           lambda: oracle.ref_softmax_f32(x, axis))


@pytest.mark.parametrize("op,coeff", [(2, (1.0, 1.0)), (2, (0.5, -1.5)), (1, (1.0, 1.0)), (3, (1.0, 1.0))])   # sum, prod, max
@pytest.mark.parametrize("relu", [False, True])
def test_eltwise_matches_reference_test_oracle(oracle, reference, op, coeff, relu):
    rng = np.random.default_rng(op * 7 + int(relu))
    a = rng.uniform(-2, 2, 4099).astype(np.float32)
    b = rng.uniform(-2, 2, 4099).astype(np.float32)
    reference.assert_equal("eltwise%r" % ((op, coeff, relu),), oracle.eltwise_f32(a, b, op, coeff[0], coeff[1], relu),
                           lambda: oracle.ref_eltwise_f32(a, b, op, coeff[0], coeff[1], relu))


@pytest.mark.parametrize("act,coef", [(2, 1.0), (1, 1.0), (3, 1.0), (4, 1.5), (5, 0.7)])   # relu sigmoid tanh clipped elu
def test_activation_matches_reference_test_oracle(oracle, reference, act, coef):
    x = np.random.default_rng(act).uniform(-4, 4, (2, 3, 5, 7)).astype(np.float32)
    reference.assert_equal("activation%r" % ((act, coef),), oracle.activation_f32(x, act, 0.0, coef),
                           lambda: oracle.ref_activation_f32(x, act, 0.0, coef))


def test_grouped_x86_int8_conv_agrees_with_reference_oracle_on_shared_subset(oracle, reference):
    """Depthwise / grouped INT8: the grouped x86 restatement coincides with the reference's own conv_basic_check_int8
    (which takes `group`) on their shared subset -- integral bias, s8 output, no residual."""
    rng = np.random.default_rng(23)
    for c, k, group in ((16, 16, 16), (32, 32, 32), (16, 32, 4)):
        x = rng.integers(-128, 128, (2, 9, 9, c)).astype(np.int8)
        w = rng.integers(-127, 128, (k, c // group, 3, 3)).astype(np.int8)
        b = rng.integers(-1000, 1000, k).astype(np.int32)
        sc = rng.uniform(0.002, 0.02, k).astype(np.float32)
        for relu in (False, True):
            j = oracle.conv_s8_nhwc_x86(x, w, b.astype(np.float32), sc, pad=(1, 1), stride=(2, 2), relu=relu,
                                        out_dtype=oracle.DT_INT8, group=group)
            reference.assert_equal("conv_int8_basic grouped%r" % ((c, k, group, relu),), j,
                                   lambda: oracle.conv_s8_nhwc_basic(x, w, b, sc, pad=(1, 1), stride=(2, 2), relu=relu,
                                                                     group=group, use_ref=True))
    # group == 1 through the grouped entry point is the ungrouped function
    x = rng.integers(0, 256, (1, 7, 7, 16)).astype(np.uint8)
    w = rng.integers(-127, 128, (8, 16, 3, 3)).astype(np.int8)
    sc = rng.uniform(0.002, 0.02, 8).astype(np.float32)
    a = oracle.conv_s8_nhwc_x86(x, w, None, sc, out_dtype=oracle.DT_UINT8, relu=True)
    import ctypes as C
    out = np.zeros_like(a)
    oracle.lib().oracle_conv_s8_nhwc_x86_group(oracle._p(x), oracle._dt(x), oracle._p(w), None, oracle._p(sc), None, -1,
                                               oracle._f(1.0), oracle._p(out), oracle.DT_UINT8, 1, 16, 7, 7, 8, 1, 3, 3,
                                               1, 1, 1, 1, 0, 0, 1)
    np.testing.assert_array_equal(out, a)


def test_fast_fp32_conv_equals_the_scalar_restatement_up_to_reassociation(oracle):
    """oracle_conv_f32_nhwc_packed (the CPU-baseline arm's AVX-512 fp32 convolution: same sums, fused multiply-adds) against
    oracle_conv_f32_nhwc with the reference's own criterion (tensor_cmp_host) at 1e-5 -- 100x tighter than the 1e-3 the parity
    tests apply to the GPU path; and the walker on top of it against the committed fp32 goldens."""
    if not oracle.vnni_available():
        pytest.skip("no AVX-512 on this CPU")
    rng = np.random.default_rng(5)
    for (n, h, w, c, k, r, st, pad, dil) in [(2, 14, 14, 64, 72, 3, 1, 1, 1), (1, 9, 11, 16, 40, 3, 2, 1, 2), (3, 7, 7, 128, 130, 1, 1, 0, 1),
                                             (1, 20, 20, 3, 64, 7, 2, 3, 1), (4, 1, 1, 512, 100, 1, 1, 0, 1), (1, 5, 5, 8, 10, 3, 1, 1, 1)]:
        x = rng.uniform(-1, 1, (n, h, w, c)).astype(np.float32)
        wt = (rng.standard_normal((k, c, r, r)) * np.sqrt(2.0 / (c * r * r))).astype(np.float32)
        b = rng.uniform(-0.5, 0.5, k).astype(np.float32)
        oh, ow = oracle.conv_out_size(h, pad, dil, r, st), oracle.conv_out_size(w, pad, dil, r, st)
        res = rng.uniform(-1, 1, (n, oh, ow, k)).astype(np.float32)
        for rs, bias, relu in ((None, b, True), (res, b, True), (res, None, False)):
            kw = dict(residual=rs, stride=(st, st), pad=(pad, pad), dil=(dil, dil), relu=relu, neg_slope=0.1, beta=1.0)
            want = oracle.conv_f32_nhwc(x, wt, bias, **kw)
            got = oracle.conv_f32_nhwc(x, wt, bias, fast=True, **kw)
            mr, md = oracle.tensor_cmp(want, got)
            assert md < 1e-5 or mr <= 1e-5, ((n, h, w, c, k, r), mr, md)
    from anakin_b200 import modelzoo
    from oracle import model_walker as W
    gold = np.load(os.path.join(GOLD, "tiny_resnet_golden.npz"))
    g = modelzoo.build("tiny_resnet", batch=1)
    cache = {}
    for _ in range(2):
        _, vals = W.run_fp32(g, modelzoo.synthetic_input(4, 32), return_values=True, fast=True, weight_cache=cache)
        mr, md = oracle.tensor_cmp(gold["logits_fp32"][:4], vals["fc"].reshape(4, -1))
        assert md < 1e-4 or mr <= 1e-4, (mr, md)


def test_fast_int8_pooling_is_bit_identical_to_the_scalar_restatement(oracle):
    """oracle_pool_s8_nhwc_fast (the CPU-baseline arm's AVX-512 pooling) == oracle_pool_s8_nhwc: max / avg incl. / avg excl.
    padding, s8 and u8 codes, padded and ceil-mode windows, global pooling, channel counts off the vector widths."""
    if not oracle.vnni_available():
        pytest.skip("no AVX-512 on this CPU")
    rng = np.random.default_rng(77)
    for (n, h, w, c) in [(2, 13, 17, 64), (1, 12, 12, 100), (3, 7, 7, 2048), (1, 9, 5, 8)]:
        for uns in (True, False):
            x = rng.integers(0, 256, (n, h, w, c)).astype(np.uint8) if uns else rng.integers(-128, 128, (n, h, w, c)).astype(np.int8)
            for ptype in (1, 2, 3):
                for window, pad, stride, glob in (((3, 3), (0, 0), (2, 2), False), ((3, 3), (1, 1), (2, 2), False),
                                                  ((2, 2), (0, 0), (2, 2), False), ((3, 2), (1, 0), (1, 2), False),
                                                  ((7, 7), (0, 0), (1, 1), True)):
                    a = oracle.pool_s8_nhwc(x, window, pad, stride, ptype, global_pooling=glob, fast=True)
                    b = oracle.pool_s8_nhwc(x, window, pad, stride, ptype, global_pooling=glob)
                    np.testing.assert_array_equal(a, b, err_msg=str((n, h, w, c, uns, ptype, window, pad, stride, glob)))


def test_vnni_int8_conv_is_bit_identical_to_the_scalar_restatement(oracle):
    """oracle_vnni.c (the CPU-baseline arm's AVX-512 VNNI convolution) == oracle_conv_s8_nhwc_x86 on every dtype pair,
    with / without residual, signed and unsigned inputs, channel counts that need padding, ragged tiles. Skipped where
    the CPU has no AVX-512 VNNI (the fast path then falls back to the scalar code by itself)."""
    if not oracle.vnni_available():
        pytest.skip("no AVX-512 VNNI on this CPU")
    rng = np.random.default_rng(31)
    cases = [(2, 14, 256, 72, 3, 1, 1, True), (1, 9, 16, 40, 3, 2, 1, False), (2, 20, 64, 130, 1, 1, 0, True),
             (1, 32, 3, 64, 7, 2, 3, False), (1, 7, 36, 17, 5, 1, 2, True)]
    for n, h, c, k, r, st, pad, uns in cases:
        x = (rng.integers(0, 256, (n, h, h, c)).astype(np.uint8) if uns else rng.integers(-128, 128, (n, h, h, c)).astype(np.int8))
        w = rng.integers(-127, 128, (k, c, r, r)).astype(np.int8)
        b = rng.uniform(-1000, 1000, k).astype(np.float32)
        sc = rng.uniform(0.5, 1.5, k).astype(np.float32) * np.float32(1e-3)
        oh = oracle.conv_out_size(h, pad, 1, r, st)
        res = rng.integers(0, 256, (n, oh, oh, k)).astype(np.uint8)
        for od in (oracle.DT_UINT8, oracle.DT_INT8, oracle.DT_FLOAT):
            for rs in (None, res):
                kw = dict(residual=rs, sum_scale=0.37, out_dtype=od, stride=(st, st), pad=(pad, pad), relu=od != oracle.DT_INT8)
                np.testing.assert_array_equal(oracle.conv_s8_nhwc_x86(x, w, b, sc, fast=True, **kw),
                                              oracle.conv_s8_nhwc_x86(x, w, b, sc, **kw), err_msg=str((n, h, c, k, r, od)))
    # residual dtypes (s8, fp32), sum_scale == 1 (plain add instead of the fma), dilation, fewer pixels than one register tile,
    # fewer output channels than one vector, the inner product as a 1x1 conv, no bias / no scale tables, relu into s8
    for (n, h, wd, c, k, r, st, pad, dil, res_dt, ss) in [(1, 3, 4, 8, 10, 1, 1, 0, 1, np.int8, 1.0), (2, 11, 13, 12, 33, 3, 1, 2, 2, np.float32, 1.0),
                                                          (8, 1, 1, 2048, 1000, 1, 1, 0, 1, None, 1.0), (3, 8, 5, 32, 48, 3, 2, 1, 1, np.int8, 0.61)]:
        x = rng.integers(0, 256, (n, h, wd, c)).astype(np.uint8)
        w = rng.integers(-127, 128, (k, c, r, r)).astype(np.int8)
        oh, ow = oracle.conv_out_size(h, pad, dil, r, st), oracle.conv_out_size(wd, pad, dil, r, st)
        res = None
        if res_dt is np.int8:
            res = rng.integers(-128, 128, (n, oh, ow, k)).astype(np.int8)
        elif res_dt is np.float32:
            res = rng.uniform(-50, 50, (n, oh, ow, k)).astype(np.float32)
        sc = rng.uniform(0.5, 1.5, k).astype(np.float32) * np.float32(1e-3)
        for od, bias, scale, relu in ((oracle.DT_INT8, None, sc, True), (oracle.DT_UINT8, rng.uniform(-900, 900, k).astype(np.float32), sc, False),
                                      (oracle.DT_FLOAT, None, None, False)):
            kw = dict(residual=res, sum_scale=ss, out_dtype=od, stride=(st, st), pad=(pad, pad), dil=(dil, dil), relu=relu)
            np.testing.assert_array_equal(oracle.conv_s8_nhwc_x86(x, w, bias, scale, fast=True, **kw),
                                          oracle.conv_s8_nhwc_x86(x, w, bias, scale, **kw), err_msg=str((n, h, wd, c, k, r, od)))
    # the pack of a weight array is made once and reused
    assert oracle._vnni_pack(w)[0].value == oracle._vnni_pack(w)[0].value
