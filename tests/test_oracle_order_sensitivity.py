"""Documents (and guards) a property of the REFERENCE that shapes the parity bar: its numerics are
chaotic w.r.t. f32 summation order.  The truncating Q8_0 activation quantizer (buf_q8_0.rs:118-125)
and the f16 exp LUT (cpu_device.rs:108-115) amplify 1e-7 perturbations, so the reference's own scalar
(buf_q8_0.rs:275-286) and AVX2 (buf_q8_0.rs:228-272) vec_dot orders -- both exercised by its CI
(.github/workflows/ci.yml:51-57) -- give logits that differ by percents, while the greedy text is equal.
Hence: fast GPU kernels are held to op-level parity + this band; the 1e-3 bar is proven in exact_order mode.
Measured on the Q8_0 test model of tests/synth_model.py (the reference's trained fixture gave 1.6-4.1 %)."""
import numpy as np

from oracle import oracle as oc
from oracle.llama_replay import GGUFModel, Llama2Runner, load_weights
from oracle.tensor_ref import OracleDevice, OracleTensor
from tests.test_oracle_golden_text import CASES, PROMPT_IDS


def order_band(path, n_pos=len(PROMPT_IDS)):
    gm = GGUFModel(path)
    res = []
    for flags in (0, oc.ORDER_AVX2):
        dev = OracleDevice(flags=flags)
        r = Llama2Runner(OracleTensor, gm.conf, load_weights(gm, OracleTensor, dev), dev, 200)
        res.append(np.stack([r.forward([t], p).copy() for p, t in enumerate(PROMPT_IDS[:n_pos])]))
    a, b = res
    return np.abs(a - b).max(1) / np.abs(a).max(1), a.argmax(1), b.argmax(1)


def test_reference_scalar_vs_avx2_order_band(fixture_path):
    band, am_a, am_b = order_band(fixture_path("tinyllamas-stories-15m-q8_0.gguf"))
    assert band.max() > 5e-3, "the reference's two CI legs used to differ by >1e-3 in logits"
    assert band.max() < 0.1
    # ... yet the sampled token (after the last prompt position) agrees, which is all the reference's tests
    # check; at teacher-forced positions even the argmax may flip
    assert am_a[-1] == am_b[-1] == CASES[0][2][0]
