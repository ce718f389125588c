"""Regenerates the golden data of the GGUF test models (tests/synth_model.py) with the CPU oracle.

Run:  python tests/golden/make_golden.py
1. classifier_rows.npz: for each model, the classifier rows of its golden tokens (CASES of tests/test_oracle_golden_text.py),
   fitted to the final hidden states the oracle computes on the model with random rows for the prompt followed by the
   golden tokens (synth_model.fit_rows);
2. *_synth_logits.npz: the oracle's generation on the finished models, logits at a few steps and, to keep the files small,
   at a fixed sample of vocabulary entries (COLS).
The oracle is itself pinned by the reference's KATs (tests/test_oracle_kats.py).  tinyllamas-stories-15m-*_logits.npz
(without _synth) are the oracle's outputs on the reference's trained models, kept as a record; no test reads them.
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.llama_replay import GGUFModel, Llama2Runner, load_weights  # noqa: E402
from oracle.tensor_ref import OracleDevice, OracleTensor  # noqa: E402
from tests import synth_model  # noqa: E402
from tests.conftest import find_fixture  # noqa: E402
from tests.test_oracle_golden_text import CASES, PROMPT_IDS, run_oracle  # noqa: E402

STEPS = np.array([0, 1, 5, 10])
N_COLS = 1024

fits = {}
with tempfile.TemporaryDirectory() as d:
    for fname, text, ids in CASES:
        path = os.path.join(d, fname)
        synth_model.write_model(path, fname, fitted=False)
        gm = GGUFModel(path)
        dev = OracleDevice(debug_named_tensors=True)
        r = Llama2Runner(OracleTensor, gm.conf, load_weights(gm, OracleTensor, dev), dev, 200)
        seq = PROMPT_IDS + ids[:-1]                  # teacher-forced: the positions whose logits pick ids[0], ids[1], ...
        best = [float(r.forward([t], p).max()) for p, t in enumerate(seq)][len(PROMPT_IDS) - 1:]
        hidden = np.stack([dev.debug_tensors[f"final_rmsnorm:{p}"] for p in range(len(PROMPT_IDS) - 1, len(seq))])
        key = fname[:-len(".gguf")]
        fits[f"{key}_ids"] = np.array(ids)
        fits[f"{key}_rows"] = synth_model.fit_rows(hidden, np.array(best))
np.savez_compressed(os.path.join(HERE, "classifier_rows.npz"), **fits)

for fname, text, ids in CASES:
    gm, tok, prompt_ids, out, logits, dev = run_oracle(find_fixture(fname), debug=True)
    assert out == ids, (fname, out)
    logits = np.stack(logits)[STEPS]
    cols = np.union1d(np.random.default_rng(0).choice(logits.shape[1], N_COLS, replace=False), logits.argmax(1))
    taps = {k.replace(":", "_"): v for k, v in dev.debug_tensors.items()
            if k in ("attn_rmsnorm:0:0", "x_debug:0:0", "attn_out:0:0", "ffn_out:0:0", "ffn_out:5:9", "final_rmsnorm:9")}
    np.savez_compressed(os.path.join(HERE, fname.replace(".gguf", "_synth_logits.npz")),
                        prompt_ids=np.array(prompt_ids), generated_ids=np.array(out), steps=STEPS, cols=cols,
                        logits=logits[:, cols], **taps)
    print(fname, out, repr(text), {k: v.shape for k, v in taps.items()})
