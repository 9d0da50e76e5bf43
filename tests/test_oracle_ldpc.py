"""Pin the CPU oracle (oracle/ldpc_bp_ref.c + oracle/ldpc.py) against the reference's own known-answer tests and
golden vectors (no TensorFlow needed):
  * node updates vs the NumPy loops of /root/reference/test/unit/fec/test_ldpc_decoding.py:397-654 (restated here),
    tolerance rtol = atol = 1e-3 exactly as the reference tests use; both math modes of the oracle;
  * duplicate-minimum KAT (:503-510), all-erasure KAT (:277-290, :944-959), llr_max bound (:361-376, :978-997),
    message routing with identity node functions (:53-88), rate-matching identity at 0 iterations (:1023-1040);
  * phi() values of SURVEY.md Appendix A;
  * encoder vs the 28 generator-matrix goldens (tests/golden/ldpc_enc_golden.npz, made from
    /root/reference/test/codes/ldpc/*.npy by tests/golden/make_ldpc_enc_golden.py).
"""
import os
import numpy as np
import pytest

from oracle import ldpc as O

DEGS = [3, 4, 5, 6, 7]
CLIPS = [5, 20, 100, None]
MODES = [0, 1]


def _clip(v, c):
    return v if c is None else np.maximum(np.minimum(v, c), -c)


def _rand_msgs(rng, deg, bs=100):
    return rng.normal(size=(deg, bs)).astype(np.float32) * 3.0


@pytest.mark.parametrize("clip", CLIPS)
@pytest.mark.parametrize("no", [0, 0.1, 1.0])
def test_vn_update_sum(clip, no):
    rng = np.random.default_rng(1)
    for deg in DEGS:
        msg = _rand_msgs(rng, deg)
        llr = (no * rng.normal(size=msg.shape[1])).astype(np.float32)
        x_tot_ref = msg.astype(np.float64).sum(0) + llr
        x_e_ref = x_tot_ref[None, :] - msg
        for b in range(msg.shape[1]):
            out, xt = O.vn_update("sum", msg[:, b], llr[b], clip)
            assert np.allclose(out, _clip(x_e_ref[:, b], clip), rtol=1e-3, atol=1e-3)
            assert np.allclose(xt, _clip(x_tot_ref[b], clip), rtol=1e-3, atol=1e-3)


def _minsum_ref(x, offset):
    sign_out = np.prod(np.sign(x), axis=0, keepdims=True) * np.sign(x)
    a = np.abs(x)
    out = np.zeros_like(a, dtype=np.float64)
    for i in range(a.shape[0]):
        cur = np.min(np.delete(a, i, axis=0), axis=0)
        out[i] = np.maximum(cur - offset, 0) * sign_out[i]
    return out


@pytest.mark.parametrize("clip", CLIPS)
@pytest.mark.parametrize("offset", [0, 0.5, 1.0])
def test_cn_update_offset_minsum(clip, offset):
    rng = np.random.default_rng(2)
    for deg in DEGS:
        msg = _rand_msgs(rng, deg)
        ref = _clip(_minsum_ref(msg.astype(np.float64), offset), clip)
        for b in range(msg.shape[1]):
            out = O.cn_update("offset-minsum", msg[:, b], clip, offset=offset)
            assert np.allclose(out, ref[:, b], rtol=1e-3, atol=1e-3)
            if offset == 0:
                assert np.array_equal(out, O.cn_update("minsum", msg[:, b], clip))


def test_cn_minsum_duplicate_minimum():
    out = O.cn_update("minsum", [2.1, 2.1, 3, 4], None)
    assert np.allclose(out, [2.1, 2.1, 2.1, 2.1])
    out = O.cn_update("minsum", [-2.1, 2.1, 3, -4], None)
    assert np.allclose(out, [-2.1, 2.1, 2.1, -2.1])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("clip", CLIPS)
def test_cn_update_boxplus(clip, mode):
    rng = np.random.default_rng(3)
    for deg in DEGS:
        msg = _rand_msgs(rng, deg)
        for b in range(msg.shape[1]):
            cn = msg[:, b].astype(np.float64)
            ref = np.array([2 * np.arctanh(np.prod(np.tanh(np.delete(cn, i) / 2))) for i in range(deg)])
            out = O.cn_update("boxplus", msg[:, b], clip, math_mode=mode)
            assert np.allclose(out, _clip(ref, clip), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("clip", CLIPS)
def test_cn_update_boxplus_phi(clip, mode):
    rng = np.random.default_rng(4)
    for deg in DEGS:
        msg = _rand_msgs(rng, deg)
        for b in range(msg.shape[1]):
            cn = msg[:, b].astype(np.float64)
            ref = np.zeros(deg)
            for i in range(deg):
                o = np.delete(cn, i)
                v = np.sum(-np.log(np.tanh(np.abs(o) / 2)))
                ref[i] = np.prod(np.sign(o)) * (-np.log(np.tanh(v / 2)))
            out = O.cn_update("boxplus-phi", msg[:, b], clip, math_mode=mode)
            assert np.allclose(out, _clip(ref, clip), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("mode", MODES)
def test_phi_known_values(mode):
    # SURVEY.md Appendix A (NumPy float32 evaluation of decoding.py:1110-1120)
    assert O.phi(0.0, mode) == pytest.approx(16.635532, abs=2e-6)
    assert O.phi(8.5e-8, mode) == pytest.approx(16.635532, abs=2e-6)
    assert O.phi(1.0, mode) == pytest.approx(0.7719368, abs=1e-6)
    assert O.phi(10.0, mode) == pytest.approx(9.1552734e-05, abs=2e-6)
    for x in (16.0, 16.635532, 40.0, 2 * 16.635532):
        assert O.phi(x, mode) == 0.0


def _example(i):
    p = os.path.join(os.path.dirname(O.__file__), "..", "sionna_b200", "phy", "fec", "ldpc", "codes", "example_pcms.npz")
    with np.load(p) as d:
        return d[f"pcm{i}"].astype(np.float64)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("rule", ["boxplus-phi", "boxplus", "minsum", "offset-minsum"])
def test_all_erasure_gives_exact_zero(rule, mode):
    for pid in (0, 3, 4):
        pcm = _example(pid)
        x = O.bp_decode(pcm, np.zeros((3, pcm.shape[1]), np.float32), num_iter=5, cn_update=rule, hard_out=False,
                        math_mode=mode)
        assert np.all(x == 0.0)
    enc = O.LDPC5GEncoderRef(100, 200)
    x = O.LDPC5GDecoderRef(enc, cn_update=rule, hard_out=False, num_iter=5)(np.zeros((2, 200), np.float32),
                                                                           math_mode=mode)
    assert np.all(x == 0.0)


def test_identity_nodes_route_messages():
    """With identity CN/VN functions the output is llr * (deg + 1) and every edge carries its VN's llr."""
    pcm = _example(4)
    rng = np.random.default_rng(5)
    llr = rng.normal(size=(4, pcm.shape[1])).astype(np.float32)
    x, st = O.bp_decode(pcm, llr, num_iter=1, cn_update="identity", vn_update="identity", hard_out=False,
                        llr_max=1000.0, return_state=True)
    deg = pcm.sum(0)
    assert np.allclose(x, llr * (deg + 1), rtol=1e-5, atol=1e-5)
    _, vn_idx = O.ref_edges(pcm)
    assert np.allclose(st, llr.T[vn_idx, :])


@pytest.mark.parametrize("rule", ["boxplus-phi", "boxplus", "minsum", "offset-minsum"])
def test_llr_max_bound_and_state_handover(rule):
    enc = O.LDPC5GEncoderRef(60, 150)
    rng = np.random.default_rng(6)
    llr = (rng.normal(size=(5, 150)) * 30).astype(np.float32)
    for llr_max in (5.0, 20.0):
        dec = O.LDPC5GDecoderRef(enc, cn_update=rule, hard_out=False, return_infobits=False, num_iter=6,
                                 llr_max=llr_max, return_state=True)
        x, st = dec(llr)
        assert np.abs(x).max() <= llr_max and np.abs(st).max() <= llr_max
    dec1 = O.LDPC5GDecoderRef(enc, cn_update=rule, hard_out=False, num_iter=1, return_state=True)
    x1, s1 = dec1(llr)
    for _ in range(3):
        x1, s1 = dec1(llr, msg_v2c=s1)
    x4, s4 = O.LDPC5GDecoderRef(enc, cn_update=rule, hard_out=False, num_iter=4, return_state=True)(llr)
    assert np.array_equal(x1, x4) and np.array_equal(s1, s4)


@pytest.mark.parametrize("k,n", [(12, 20), (20, 50), (30, 70), (100, 300), (500, 1000), (1000, 3000), (8448, 23000)])
def test_rate_matching_identity_at_zero_iterations(k, n):
    """0 iterations: the decoder returns the (clipped) channel logits (test_ldpc_decoding.py:1023-1040)."""
    enc = O.LDPC5GEncoderRef(k, n)
    rng = np.random.default_rng(k)
    llr = rng.normal(size=(2, n)).astype(np.float32) * 4
    x = O.LDPC5GDecoderRef(enc, hard_out=False, return_infobits=False, num_iter=0)(llr)
    assert np.array_equal(x, llr)


def test_encoder_vs_reference_generator_matrices():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ldpc_enc_golden.npz"))
    assert len(g["params"]) == 28
    for k, n in g["params"]:
        u = np.unpackbits(g[f"u_{k}_{n}"], axis=1)[:, :k]
        c = np.unpackbits(g[f"c_{k}_{n}"], axis=1)[:, :n]
        enc = O.LDPC5GEncoderRef(int(k), int(n))
        assert np.array_equal(enc(u), c.astype(np.float32)), f"k={k} n={n}"


def test_encoder_vs_full_generator_matrix_small():
    """Every row of the encoder vs the reference's whole k=64, n=128 generator matrix (stored bit-packed)."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ldpc_enc_golden.npz"))
    gm = np.unpackbits(g["g_64_128"], axis=1)[:, :128]
    assert gm.shape == (64, 128) and gm.sum() > 0
    enc = O.LDPC5GEncoderRef(64, 128)
    assert np.array_equal(enc(np.eye(64, dtype=np.int64)), gm.astype(np.float32))


@pytest.mark.parametrize("rule", ["boxplus-phi", "minsum"])
def test_e2e_error_free_and_modes_agree(rule):
    """no = 0.3 BPSK: error-free recovery (test_ldpc_decoding.py:817-846); libm / kernel-math modes and
    reference / kernel summation orders give the same bits."""
    rng = np.random.default_rng(8)
    for k, n in ((100, 334), (617, 1234), (810, 900)):
        enc = O.LDPC5GEncoderRef(k, n)
        u = rng.integers(0, 2, (8, k))
        c = enc(u)
        no = 0.3
        y = (2.0 * c - 1.0) + rng.normal(size=c.shape) * np.sqrt(no / 2)
        llr = (4 * y / no).astype(np.float32)
        dec = O.LDPC5GDecoderRef(enc, cn_update=rule, num_iter=20)
        a = dec(llr)
        b = dec(llr, math_mode=1, order="kernel")
        assert np.array_equal(a, u) and np.array_equal(b, u)
