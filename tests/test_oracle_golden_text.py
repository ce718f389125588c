"""End-to-end pin of the oracle on the GGUF test models of tests/synth_model.py (synthetic weights of the shapes of the
reference's tinyllamas-stories-15M fixtures): the prompt of the reference's generation test (crabml-llama2/src/llama2.rs:
673-719), greedy decode, and the models' own golden generations (CASES).  The reference's golden strings belong to its
trained models, which the repository does not hold."""
import os

import numpy as np
import pytest

from oracle.llama_replay import GGUFModel, Llama2Runner, LlamaTokenizer, decode_text, load_weights
from oracle.tensor_ref import OracleDevice, OracleTensor

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
PROMPT = "Lily is a cute cat, "
PROMPT_IDS = [1, 365, 2354, 338, 263, 274, 1082, 6635, 29892, 29871]

CASES = [                                                # golden generations of the test models (tests/synth_model.py)
    ("tinyllamas-stories-15m-q8_0.gguf", "$(DiecolonslBI parteStar loudпро})кт",
     [12330, 16334, 17308, 2536, 12809, 3810, 16213, 22526, 5945, 1800, 3931]),
    ("tinyllamas-stories-15m-q4_0.gguf", "ierreжива guerra månős `[ Media Farctors :)бря",
     [6349, 13204, 9798, 15186, 14773, 10338, 8213, 8413, 14359, 4248, 5542]),
]


def run_oracle(path, steps=11, f16_kv=False, debug=False):
    gm = GGUFModel(path)
    dev = OracleDevice(debug_named_tensors=debug)
    w = load_weights(gm, OracleTensor, dev)
    tok = LlamaTokenizer(gm.tokens, gm.scores, gm.bos, gm.eos)
    ids = tok.encode(PROMPT, True, False)
    r = Llama2Runner(OracleTensor, gm.conf, w, dev, 200, use_f16_kv_cache=f16_kv)
    logits = []
    pos, _, t0 = r.prefill(ids)
    logits.append(r.logits.copy())
    out = []
    for t in r.generate(pos, t0, steps, eos=gm.eos):
        out.append(t)
        logits.append(r.logits.copy())
    return gm, tok, ids, out, logits, dev


@pytest.mark.parametrize("fname,text,ids", CASES)
def test_test_model_generation_needs_the_transformer(fixture_path, tmp_path, monkeypatch, fname, text, ids):
    """The golden generation of a test model comes out with either KV cache, and only when the layers and the rotary
    embedding are computed: without what the layers add to the residual, or with RoPE as the identity, it changes."""
    from tests import synth_model
    gm, tok, prompt_ids, out, _, _ = run_oracle(fixture_path(fname))
    assert gm.conf.rope_dim == 48 and gm.conf.head_size() == 48
    assert prompt_ids == PROMPT_IDS
    assert out == ids and decode_text(tok, out) == text
    assert run_oracle(fixture_path(fname), f16_kv=True)[3] == ids
    no_layers = str(tmp_path / fname)
    synth_model.write_model(no_layers, fname, layer_gain=0.0)
    assert run_oracle(no_layers)[3] != ids
    monkeypatch.setattr(OracleTensor, "rope_inplace", lambda self, mode, pos, rope_dims: self)
    assert run_oracle(fixture_path(fname))[3] != ids


@pytest.mark.parametrize("fname", [c[0] for c in CASES])
def test_committed_logits_fixture(fixture_path, fname):
    """tests/golden/*_synth_logits.npz were produced by tests/golden/make_golden.py from the oracle on the
    GGUF test models (at a fixed sample of vocabulary entries); this guards the oracle (and the models) against drift."""
    npz = os.path.join(GOLDEN, fname.replace(".gguf", "_synth_logits.npz"))
    if not os.path.exists(npz):
        pytest.skip("golden npz not generated")
    g = np.load(npz)
    _, _, _, out, logits, _ = run_oracle(fixture_path(fname))
    assert out == g["generated_ids"].tolist()
    np.testing.assert_array_equal(np.stack(logits)[g["steps"]][:, g["cols"]], g["logits"])
