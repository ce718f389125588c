"""GGUF test models of the shapes of the reference's tinyllamas-stories-15M fixtures (named after them): the architecture
(dim 288, 6 layers of 6 heads of 48, hidden 768, vocabulary 32000, context 256), tensor names and types (Q8_0 / Q4_0) and
the Llama tokenizer of the published files, with synthetic weights from a fixed seed instead of the trained ones, so that
every test that loads a GGUF model runs from the repository alone.  The vocabulary is stored in tests/golden/llama_vocab.npz
(token bytes, delta-coded integer scores, token types); the files are written on first use to a directory under the
system temporary directory.

All weights are synthetic at full scale, except the classifier rows of the golden tokens (CASES of
tests/test_oracle_golden_text.py, drawn at random).  Those rows were fitted once (tests/golden/make_golden.py) to the
final hidden states the oracle computes for the prompt followed by the golden tokens, and are stored in
tests/golden/classifier_rows.npz: row k scores hidden state k at MARGIN times the best random row and the other fitted
states at zero.  So the greedy generation is the golden one only if the transformer reproduces those hidden states --
removing the layers or the rotary embedding changes it (tests/test_oracle_golden_text.py) -- while summation-order noise
does not."""
from __future__ import annotations

import hashlib
import os
import tempfile

import numpy as np

from crabml_b200.runner import synth_scale
from oracle import oracle as oc
from oracle.synth import synth_weight

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
SEED = 0x15F
MARGIN = 1.3

DIM, HIDDEN, LAYERS, HEADS, VOCAB, CONTEXT = 288, 768, 6, 6, 32000, 256
MODELS = {"tinyllamas-stories-15m-q8_0.gguf": oc.Q8_0, "tinyllamas-stories-15m-q4_0.gguf": oc.Q4_0}
# every file the written models depend on
INPUTS = ["tests/synth_model.py", "tests/golden/llama_vocab.npz", "tests/golden/classifier_rows.npz", "oracle/synth.py",
          "oracle/crabml_oracle.c", "crabml_b200/runner.py"]


def load_vocab():
    v = np.load(os.path.join(GOLDEN, "llama_vocab.npz"))
    ends = np.cumsum(v["lengths"].astype(np.int64))
    blob = v["tokens"].tobytes()
    tokens = [blob[e - n:e] for e, n in zip(ends, v["lengths"].astype(np.int64))]
    return tokens, np.cumsum(v["score_deltas"].astype(np.int64)).astype(np.float32), v["token_type"]


def fitted_rows(name):
    """-> (token ids, float32 rows [n, DIM]): the fitted classifier rows of model `name`."""
    g = np.load(os.path.join(GOLDEN, "classifier_rows.npz"))
    key = name[:-len(".gguf")]
    return g[f"{key}_ids"], g[f"{key}_rows"]


def model_path(name: str) -> str:
    """Path of the model `name` (a key of MODELS), written on first use."""
    h = hashlib.sha1()
    for f in INPUTS:
        with open(os.path.join(ROOT, f), "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), f"crabml-b200-test-models-{os.getuid()}-{h.hexdigest()[:12]}")
    path = os.path.join(d, name)
    if not os.path.exists(path):
        os.makedirs(d, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        write_model(tmp, name)
        os.replace(tmp, path)          # concurrent test processes never see a partial file
    return path


def write_model(path: str, name: str, layer_gain: float = 1.0, fitted: bool = True) -> None:
    """layer_gain scales the attention and FFN output projections (0 removes what the layers add to the residual);
    fitted=False leaves every classifier row random (the model the rows are fitted on)."""
    import gguf
    import gguf.quants
    wt = MODELS[name]
    qt = gguf.GGMLQuantizationType(wt)
    tokens, scores, token_type = load_vocab()
    w = gguf.GGUFWriter(path, "llama")
    w.add_name(name[:-len(".gguf")])
    w.add_context_length(CONTEXT)
    w.add_embedding_length(DIM)
    w.add_block_count(LAYERS)
    w.add_feed_forward_length(HIDDEN)
    w.add_rope_dimension_count(DIM // HEADS)
    w.add_head_count(HEADS)
    w.add_head_count_kv(HEADS)
    w.add_layer_norm_rms_eps(1e-5)
    w.add_tokenizer_model("llama")
    w.add_token_list(tokens)
    w.add_token_scores(scores.tolist())
    w.add_token_types(token_type.tolist())
    w.add_bos_token_id(1)
    w.add_eos_token_id(2)
    w.add_unk_token_id(0)
    rng = np.random.default_rng([SEED, wt])
    tid = [0]

    def quant(tname, rows, cols, gain=1.0):
        tid[0] += 1
        raw = synth_weight(wt, rows, cols, SEED, tid[0], gain * synth_scale(wt, cols)).reshape(rows, -1)
        # negate the f16 scale of a random half of the blocks: Q4_0 quants (q - 8) have mean -0.5, which would otherwise add
        # one common direction to every product and make the hidden states of all positions nearly collinear
        blocks = raw.reshape(-1, oc.block_bytes(wt))
        blocks[:, 1] ^= (np.random.default_rng([SEED, wt, tid[0]]).random(len(blocks)) < 0.5).astype(np.uint8) << 7
        if tname == "output.weight" and fitted:
            ids, frows = fitted_rows(name)
            raw[ids] = gguf.quants.quantize(frows, qt)
        w.add_tensor(tname, raw.reshape(-1), raw_shape=list(raw.shape), raw_dtype=qt)

    def norm(tname):
        w.add_tensor(tname, (1.0 + 0.05 * rng.standard_normal(DIM)).astype(np.float32))
    quant("token_embd.weight", VOCAB, DIM)
    for l in range(LAYERS):
        for t in ("attn_q", "attn_k", "attn_v"):
            quant(f"blk.{l}.{t}.weight", DIM, DIM)
        quant(f"blk.{l}.attn_output.weight", DIM, DIM, layer_gain)
        quant(f"blk.{l}.ffn_gate.weight", HIDDEN, DIM)
        quant(f"blk.{l}.ffn_down.weight", DIM, HIDDEN, layer_gain)
        quant(f"blk.{l}.ffn_up.weight", HIDDEN, DIM)
        norm(f"blk.{l}.attn_norm.weight")
        norm(f"blk.{l}.ffn_norm.weight")
    norm("output_norm.weight")
    quant("output.weight", VOCAB, DIM)
    w.write_header_to_file()
    w.write_kv_data_to_file()
    w.write_tensors_to_file()
    w.close()


def fit_rows(hidden: np.ndarray, best_random: np.ndarray) -> np.ndarray:
    """Rows R with R[k] . hidden[k] = MARGIN * best_random[k] and R[k] . hidden[j] = 0 for j != k (least-norm solution)."""
    return (np.linalg.pinv(hidden.astype(np.float64)).T * (MARGIN * best_random.astype(np.float64))[:, None]).astype(np.float32)
