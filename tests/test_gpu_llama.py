"""End-to-end parity on the GGUF test models (stand-ins for the reference's fixtures, tests/synth_model.py): the Llama2Runner replay
(llama2.rs:184-281,527-638) over CudaTensor vs the same replay over the CPU oracle.
north_star: logits within 1e-3 relative; the test models' golden generations (tests/test_oracle_golden_text.py) reproduced."""
import numpy as np
import pytest

from oracle.llama_replay import GGUFModel, Llama2Runner, LlamaTokenizer, decode_text, load_weights
from oracle.tensor_ref import OracleDevice, OracleTensor
from tests.gpu_common import make_device
from tests.test_oracle_golden_text import CASES, PROMPT, PROMPT_IDS

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3      # north_star bar (relative to max |logit|); met -- with equality -- in exact_order mode


def _band():
    # the q4_0 fixture has 9 blocks/row, where the reference's Q4_0 AVX2 kernel falls back to the scalar loop
    # (buf_q4_0.rs:220-223), so the band is taken on the q8_0 twin of the same model
    from tests.conftest import find_fixture
    from tests.test_oracle_order_sensitivity import order_band
    return float(order_band(find_fixture("tinyllamas-stories-15m-q8_0.gguf"))[0].max())


def _run(T, dev, gm, steps, f16_kv=False):
    w = load_weights(gm, T, dev)
    r = Llama2Runner(T, gm.conf, w, dev, 200, use_f16_kv_cache=f16_kv)
    logits = []
    pos, _, t0 = r.prefill(PROMPT_IDS)
    logits.append(r.logits.copy())
    out = []
    for t in r.generate(pos, t0, steps, eos=gm.eos):
        out.append(t)
        logits.append(r.logits.copy())
    return out, np.stack(logits)


@pytest.mark.parametrize("fname,text,ids", CASES)
@pytest.mark.parametrize("f16_kv", [False, True])
def test_exact_order_mode_is_bit_identical(fixture_path, fname, text, ids, f16_kv):
    """exact_order: every reduction in the reference's scalar order -> logits and every debug tap are
    BIT-IDENTICAL to the scalar CPU path, at every step (far inside the 1e-3 bar)."""
    from crabml_b200 import CudaTensor
    gm = GGUFModel(fixture_path(fname))
    tok = LlamaTokenizer(gm.tokens, gm.scores, gm.bos, gm.eos)
    assert tok.encode(PROMPT, True, False) == PROMPT_IDS
    gdev = make_device(debug_named_tensors=True, exact_order=True)
    odev = OracleDevice(debug_named_tensors=True)
    try:
        g_out, g_logits = _run(CudaTensor, gdev, gm, 11, f16_kv)
        o_out, o_logits = _run(OracleTensor, odev, gm, 11, f16_kv)
        assert g_out == o_out
        if not f16_kv or "q8_0" in fname:                     # golden generation
            assert g_out == ids and decode_text(tok, g_out) == text
        rel = (np.abs(g_logits - o_logits) / np.abs(o_logits).max(axis=1, keepdims=True)).max()
        assert rel < REL_TOL, rel
        np.testing.assert_array_equal(g_logits.view(np.uint32), o_logits.view(np.uint32))
        # debug taps: the mechanism of the reference's own cross-backend test (llama2.rs:768-784)
        for name in ("attn_rmsnorm:0:0", "x_debug:0:0", "attn_out:0:0", "ffn_out:0:0", "ffn_out:5:9", "final_rmsnorm:9"):
            a, b = gdev.dump_debug_tensor(name), odev.dump_debug_tensor(name)
            assert a is not None and a.shape == b.shape, name
            np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32), err_msg=name)
    finally:
        gdev.close()


@pytest.mark.parametrize("fname,text,ids", CASES)
def test_fast_mode_generation_and_band(fixture_path, fname, text, ids):
    """Fast (warp-parallel) kernels: same greedy text as the golden generation, and logits no
    further from the scalar reference path than the reference's own AVX2 path is (order band)."""
    from crabml_b200 import CudaTensor
    path = fixture_path(fname)
    gm = GGUFModel(path)
    tok = LlamaTokenizer(gm.tokens, gm.scores, gm.bos, gm.eos)
    gdev = make_device(debug_named_tensors=True)
    odev = OracleDevice(debug_named_tensors=True)
    try:
        g_out, g_logits = _run(CudaTensor, gdev, gm, 11)
        o_out, o_logits = _run(OracleTensor, odev, gm, 11)
        assert g_out == o_out == ids and decode_text(tok, g_out) == text
        rel = (np.abs(g_logits - o_logits) / np.abs(o_logits).max(axis=1, keepdims=True)).max()
        band = _band()
        print(f"{fname}: fast-mode max rel logits diff {rel:.3e}; reference scalar-vs-AVX2 band {band:.3e}")
        assert rel <= 1.5 * band, (rel, band)
        # before any re-quantisation of perturbed values the agreement is at f32 rounding level
        for name, eps in (("attn_rmsnorm:0:0", 1e-6), ("x_debug:0:0", 1e-6), ("attn_out:0:0", 1e-6)):
            a, b = gdev.dump_debug_tensor(name), odev.dump_debug_tensor(name)
            np.testing.assert_allclose(a, b, atol=eps * max(1.0, float(np.abs(b).max())), err_msg=name)
    finally:
        gdev.close()


def test_long_decode_positions(fixture_path):
    """100 decode steps (BASELINE config 1/2): positions up to ~110 exercise the RoPE recurrence and
    a growing KV cache; logits must stay within the bar at every step."""
    from crabml_b200 import CudaTensor
    gm = GGUFModel(fixture_path("tinyllamas-stories-15m-q8_0.gguf"))
    gdev = make_device(exact_order=True)
    try:
        g_out, g_logits = _run(CudaTensor, gdev, gm, 100)
        o_out, o_logits = _run(OracleTensor, OracleDevice(), gm, 100)
        assert g_out == o_out
        np.testing.assert_array_equal(g_logits.view(np.uint32), o_logits.view(np.uint32))
    finally:
        gdev.close()
