"""The C++ Llama2Runner replay (crabml_b200/csrc/host/llama2_runner.cpp, the product's host side) end to end:
golden generations of the GGUF test models, bit-identical logits in exact_order mode, and a
Llama-2-7B-SHAPED layer on the synthetic weights bench.py uses (BASELINE.json configs 2-4 at full size)."""
import os

import numpy as np
import pytest

from oracle import oracle as oc
from oracle.llama_replay import GGUFModel, Llama2Runner, LlamaConfig as OConf, LlamaTokenizer, LlamaWeights, decode_text, load_weights
from oracle.synth import synth_weight
from oracle.tensor_ref import OracleDevice, OracleTensor
from tests.gpu_common import make_device
from tests.test_oracle_golden_text import CASES, PROMPT_IDS

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("fname,text,ids", CASES)
@pytest.mark.parametrize("exact", [False, True])
def test_cpp_runner_golden_generation(fixture_path, fname, text, ids, exact):
    from crabml_b200 import runner as R
    path = fixture_path(fname)
    dev = make_device(exact_order=exact)
    try:
        conf, w, tok = R.load_gguf(path, dev)
        assert conf.rope_dim == 48 and conf.head_size() == 48
        r = R.LlamaRunner(dev, conf, w, 200)
        out = r.generate_greedy(PROMPT_IDS, 11, eos=tok["eos"])
        assert out == ids
        t = LlamaTokenizer(tok["tokens"], tok["scores"], tok["bos"], tok["eos"])
        assert decode_text(t, out) == text
        assert r.kv_cache_len() == len(PROMPT_IDS) + 10
        r.close()
    finally:
        dev.close()


@pytest.mark.parametrize("f16_kv", [False, True])
def test_cpp_runner_exact_logits_bit_identical(fixture_path, f16_kv):
    from crabml_b200 import runner as R
    path = fixture_path("tinyllamas-stories-15m-q8_0.gguf")
    gm = GGUFModel(path)
    odev = OracleDevice()
    ro = Llama2Runner(OracleTensor, gm.conf, load_weights(gm, OracleTensor, odev), odev, 64, use_f16_kv_cache=f16_kv)
    dev = make_device(exact_order=True)
    try:
        conf, w, _ = R.load_gguf(path, dev)
        r = R.LlamaRunner(dev, conf, w, 64, f16_kv=f16_kv)
        for pos, t in enumerate(PROMPT_IDS + [29941, 2440]):
            a = r.forward([t], pos).copy()
            b = ro.forward([t], pos)
            np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32), err_msg=f"pos {pos}")
        r.close()
    finally:
        dev.close()


@pytest.mark.parametrize("wt,ct", [(oc.Q8_0, oc.Q8_0), (oc.Q4_0, oc.Q6_K), (oc.Q4_K, oc.Q6_K)])
def test_llama2_7b_shaped_layer_on_synthetic_weights(wt, ct):
    """Full Llama-2-7B dimensions (4096 / 11008 / 32 heads / vocab 32000) with ONE layer: the synthetic weights
    are generated on the device; the oracle runs on the bit-identical CPU twin.  exact_order -> equality;
    fast mode -> within the order-noise budget of a single layer."""
    from crabml_b200 import runner as R
    conf = R.LlamaConfig(32, 32, 1, 4096, 11008, 4096, 32000, 1e-5, 128)
    seed = 0x5EED
    odev = OracleDevice()
    dim, hid = conf.embedding_dim, conf.hidden_dim

    def syn(rows, cols, t, tid):
        return OracleTensor.from_cpu(synth_weight(t, rows, cols, seed, tid, R.synth_scale(t, cols)), [rows, cols], t, odev)
    rng = np.random.default_rng(seed)

    def norm():
        return OracleTensor.from_cpu((1.0 + 0.05 * rng.standard_normal(dim)).astype(np.float32), [dim], oc.F32, odev)
    ra, rf = norm(), norm()
    lw = LlamaWeights(token_embed=syn(conf.vocab_size, dim, wt, 8), wq=[syn(dim, dim, wt, 1)], wk=[syn(dim, dim, wt, 2)],
                      wv=[syn(dim, dim, wt, 3)], wo=[syn(dim, dim, wt, 4)], ffn_gate_weight=[syn(hid, dim, wt, 5)],
                      ffn_down_weight=[syn(dim, hid, wt, 7)], ffn_up_weight=[syn(hid, dim, wt, 6)], rms_att_weight=[ra],
                      rms_ffn_weight=[rf], rms_final_weight=norm(), output_weight=syn(conf.vocab_size, dim, ct, 9))
    oconf = OConf(32, 32, 1, dim, hid, 4096, 32000, 1e-5, 128)
    ro = Llama2Runner(OracleTensor, oconf, lw, odev, 8)
    want = [ro.forward([t], p).copy() for p, t in enumerate([1, 777, 31999])]
    for exact in (True, False):
        dev = make_device(exact_order=exact)
        try:
            w = R.synthetic_weights(dev, conf, wt, ct, seed=seed)
            r = R.LlamaRunner(dev, conf, w, 8)
            for p, t in enumerate([1, 777, 31999]):
                got = r.forward([t], p).copy()
                assert np.isfinite(got).all() and np.abs(got).max() > 1e-3
                if exact:
                    np.testing.assert_array_equal(got.view(np.uint32), want[p].view(np.uint32))
                else:
                    rel = np.abs(got - want[p]).max() / np.abs(want[p]).max()
                    assert rel < 2e-2, rel          # one layer of order noise through truncating quantisers
            r.close()
        finally:
            dev.close()


@pytest.mark.parametrize("fname,text,ids", CASES)
@pytest.mark.parametrize("f16_kv", [False, True])
@pytest.mark.parametrize("mode", [1, 2])
def test_lazy_fused_graph_mode_golden_generation(fixture_path, fname, text, ids, f16_kv, mode):
    """lazy mode: same C-ABI calls, recorded -> fused kernels -> CUDA-graph replay.  Golden text, logits inside the
    reference's own order band, and the graph is actually replayed (not re-captured every token)."""
    from crabml_b200 import runner as R
    from tests.test_gpu_llama import _band
    path = fixture_path(fname)
    gm = GGUFModel(path)
    odev = OracleDevice()
    ro = Llama2Runner(OracleTensor, gm.conf, load_weights(gm, OracleTensor, odev), odev, 64, use_f16_kv_cache=f16_kv)
    dev = make_device(lazy=mode)          # 1 = fused kernels in a CUDA graph, 2 = one persistent megakernel per token
    try:
        conf, w, tok = R.load_gguf(path, dev)
        r = R.LlamaRunner(dev, conf, w, 64, f16_kv=f16_kv)
        worst = 0.0
        seq = PROMPT_IDS + ids[:6]
        for pos, t in enumerate(seq):
            a = r.forward([t], pos).copy()
            b = ro.forward([t], pos)
            worst = max(worst, float(np.abs(a - b).max() / np.abs(b).max()))
        assert worst <= 1.5 * _band(), worst
        st = dev.lazy_stats()
        assert st["uncached"] == 0, st                       # every op of the decode layer was fused or graph-safe
        assert st["graph_replays"] >= len(seq) - 4, st       # at most a few captures while the pool warms up
        r.close()
        r2 = R.LlamaRunner(dev, conf, w, 64, f16_kv=f16_kv)
        out = r2.generate_greedy(PROMPT_IDS, 11, eos=tok["eos"])
        if not f16_kv or "q8_0" in fname:
            assert out == ids
        r2.close()
    finally:
        dev.close()


def test_lazy_mode_matches_eager_ops_through_python_mirror(fixture_path):
    """The recorder is transparent for arbitrary call sequences: the Python replay (not the C++ runner), with debug
    taps forcing flushes at odd places, gives the golden generation."""
    from crabml_b200 import CudaTensor
    path = fixture_path("tinyllamas-stories-15m-q8_0.gguf")
    gm = GGUFModel(path)
    dev = make_device(lazy=True, debug_named_tensors=True)
    try:
        r = Llama2Runner(CudaTensor, gm.conf, load_weights(gm, CudaTensor, dev), dev, 64)
        pos, _, t0 = r.prefill(PROMPT_IDS)
        out = list(r.generate(pos, t0, 11, eos=gm.eos))
        assert out == CASES[0][2]
        assert dev.dump_debug_tensor("final_rmsnorm:9") is not None
    finally:
        dev.close()


@pytest.mark.parametrize("wt,ct", [(oc.Q8_0, oc.Q8_0), (oc.Q4_0, oc.Q6_K), (oc.Q4_K, oc.Q6_K)])
def test_lazy_7b_shaped_layer(wt, ct):
    """Every execution mode on the same model.  The K-quant rows do not take the streaming kernel: they check that the fuser
    hands the f32 normalised row (not only the Q8_0 scratch) to matvecs that fall back to their eager kernels."""
    from crabml_b200 import runner as R
    conf = R.LlamaConfig(32, 32, 2, 4096, 11008, 4096, 32000, 1e-5, 128)
    res = {}
    for lazy in (0, 1, 2):
        dev = make_device(lazy=lazy)
        try:
            w = R.synthetic_weights(dev, conf, wt, ct, seed=7)
            r = R.LlamaRunner(dev, conf, w, 16)
            res[lazy] = np.stack([r.forward([t], p).copy() for p, t in enumerate([1, 777, 31999, 5, 6])])
            if lazy:
                st = dev.lazy_stats()
                assert st["uncached"] == 0 and st["graph_replays"] >= 2, st
            r.close()
        finally:
            dev.close()
    # Every mode reduces with the same grouping (canonical orders, csrc/common.cuh): the recorded/fused kernels and the megakernel
    # are BIT-IDENTICAL to the eager per-op kernels, which tests/test_gpu_matvec.py and test_gpu_ops.py pin to the oracle within
    # 1e-6 * sum|terms| -- so those bounds cover the benchmarked megakernel by transitivity.
    assert np.isfinite(res[0]).all() and np.abs(res[0]).max() > 1e-3
    for mode in (1, 2):
        np.testing.assert_array_equal(res[mode].view(np.uint32), res[0].view(np.uint32), err_msg=f"lazy={mode} vs eager")


@pytest.mark.parametrize("wt,ct", [(oc.Q8_0, oc.Q8_0), (oc.Q4_0, oc.Q6_K)])
def test_both_persistent_kernels_bit_identical_on_7b_shapes(tmp_path, wt, ct):
    """The two persistent kernels -- weights through registers (mega.cu: what sharded runs and shapes the ring cannot feed use) and
    weights through the TMA-fed shared-memory ring (mega_ring.cu: the default) -- against the eager kernels on the same 7B-shaped
    model, each in its own process (the flag word that selects the kernel is read once per process)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    got = {}
    for name, lazy, flags in (("eager", 0, None), ("registers", 2, "0x4d"), ("ring", 2, None)):
        env = dict(os.environ)
        env.pop("CRABML_MEGA_FLAGS", None)
        if flags:
            env["CRABML_MEGA_FLAGS"] = flags
        out = str(tmp_path / f"{name}.npz")
        subprocess.run([sys.executable, os.path.join(root, "tests", "mega_variant_worker.py"), str(lazy), str(wt), str(ct), out],
                       check=True, cwd=root, env=env, timeout=600)
        got[name] = np.load(out)
    assert int(got["registers"]["variant"]) == 1 and int(got["ring"]["variant"]) == 2
    ref = got["eager"]["logits"]
    assert np.isfinite(ref).all() and np.abs(ref).max() > 1e-3
    for name in ("registers", "ring"):
        np.testing.assert_array_equal(got[name]["logits"].view(np.uint32), ref.view(np.uint32), err_msg=f"{name} vs eager")


@pytest.mark.parametrize("fname", ["tinyllamas-stories-15m-q8_0.gguf", "tinyllamas-stories-15m-q4_0.gguf"])
@pytest.mark.parametrize("f16_kv", [False, True])
def test_execution_modes_bit_identical_on_fixture(fixture_path, fname, f16_kv):
    """eager / CUDA-graph / megakernel on the GGUF test models (head_dim 48: unquantised attention output path,
    rows of 288 and 768: ragged last group), 24 positions so the softmax spans more than one warp."""
    from crabml_b200 import runner as R
    path = fixture_path(fname)
    seq = (PROMPT_IDS + CASES[0][2])[:21] + [5, 6, 7]
    res = {}
    for lazy in (0, 1, 2):
        dev = make_device(lazy=lazy)
        try:
            conf, w, _ = R.load_gguf(path, dev)
            r = R.LlamaRunner(dev, conf, w, 64, f16_kv=f16_kv)
            res[lazy] = np.stack([r.forward([t], p).copy() for p, t in enumerate(seq)])
            r.close()
        finally:
            dev.close()
    for mode in (1, 2):
        np.testing.assert_array_equal(res[mode].view(np.uint32), res[0].view(np.uint32), err_msg=f"lazy={mode} vs eager")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_device_side_greedy_loop_equals_the_host_sampled_loop(fixture_path, mode):
    """ccr_runner_generate_greedy_ex (sampling on the device, the id feeds the next step from a device slot, no host wait per step)
    against the plain loop forward -> export -> host argmax (sampler.rs:109-116): same ids, and the asynchronously exported logits of
    every generated position are bit-identical to the synchronously exported ones."""
    from crabml_b200 import runner as R
    path = fixture_path("tinyllamas-stories-15m-q8_0.gguf")
    dev = make_device(lazy=mode)
    try:
        conf, w, tok = R.load_gguf(path, dev)
        steps = 12
        r = R.LlamaRunner(dev, conf, w, 64)
        ids, logits = r.generate_greedy_logits(PROMPT_IDS, steps)
        assert len(ids) == steps and logits.shape == (steps, conf.vocab_size)
        assert r.kv_cache_len() == len(PROMPT_IDS) + steps - 1
        r.close()
        r2 = R.LlamaRunner(dev, conf, w, 64)
        pos, want_ids, want_logits = 0, [], []
        for t in PROMPT_IDS:
            lg = r2.forward([t], pos).copy(); pos += 1
        for _ in range(steps):
            nxt = int(np.flatnonzero(lg == lg.max())[-1])
            want_ids.append(nxt); want_logits.append(lg)
            if len(want_ids) == steps:
                break
            lg = r2.forward([nxt], pos).copy(); pos += 1
        r2.close()
        assert ids == want_ids
        np.testing.assert_array_equal(logits.view(np.uint32), np.stack(want_logits).view(np.uint32))
        assert ids[:11] == CASES[0][2]                      # and they are the golden generation
    finally:
        dev.close()


def test_fast_mode_logits_inside_the_reference_order_band_on_7b_shapes():
    """The benchmarked configuration (megakernel, warp-parallel reductions) on Llama-2-7B SHAPES, 8 layers, 32 decode positions:
    per position, the distance of the GPU logits from the reference's AVX2-order logits is compared with the distance between the
    reference's OWN two code paths (scalar vs AVX2 order, both restated in the oracle, both passing every KAT) on the same weights.
    The truncating activation quantiser (buf_q8_0.rs:117-126) makes logits chaotic in the summation order (DESIGN.md section 2), so the
    band of the reference itself is the meaningful yardstick; the distribution over the 32 positions is printed."""
    import os
    from crabml_b200 import runner as R
    nl = 8
    conf = R.LlamaConfig(32, 32, nl, 4096, 11008, 4096, 32000, 1e-5, 128)
    seed, wt = 0x5EED, oc.Q8_0
    rng = np.random.default_rng(5)
    toks = [int(t) for t in rng.integers(1, 32000, 32)]
    threads = max(1, min(16, len(os.sched_getaffinity(0))))
    logits = {}
    for name, flags in (("avx2", oc.ORDER_AVX2), ("scalar", 0)):
        odev = OracleDevice(thread_num=threads, flags=flags)
        tid = [0]

        def syn(rows, cols):
            tid[0] += 1
            return OracleTensor.from_cpu(synth_weight(wt, rows, cols, seed, tid[0], R.synth_scale(wt, cols)), [rows, cols], wt, odev)
        nrng = np.random.default_rng(seed)

        def norm():
            return OracleTensor.from_cpu((1.0 + 0.05 * nrng.standard_normal(4096)).astype(np.float32), [4096], oc.F32, odev)
        lw = LlamaWeights(None, [], [], [], [], [], [], [], [], [], None, None)
        for _ in range(nl):           # tensor ids in the order runner.synthetic_weights hands them out
            lw.wq.append(syn(4096, 4096)); lw.wk.append(syn(4096, 4096)); lw.wv.append(syn(4096, 4096)); lw.wo.append(syn(4096, 4096))
            lw.ffn_gate_weight.append(syn(11008, 4096)); lw.ffn_up_weight.append(syn(11008, 4096)); lw.ffn_down_weight.append(syn(4096, 11008))
            lw.rms_att_weight.append(norm()); lw.rms_ffn_weight.append(norm())
        lw.token_embed = syn(32000, 4096)
        lw.output_weight = syn(32000, 4096)
        lw.rms_final_weight = norm()
        ro = Llama2Runner(OracleTensor, OConf(32, 32, nl, 4096, 11008, 4096, 32000, 1e-5, 128), lw, odev, 40)
        logits[name] = np.stack([ro.forward([t], p).copy() for p, t in enumerate(toks)])
        del ro, lw
    dev = make_device(lazy=2)
    try:
        w = R.synthetic_weights(dev, conf, wt, wt, seed=seed)
        r = R.LlamaRunner(dev, conf, w, 40)
        logits["gpu"] = np.stack([r.forward([t], p).copy() for p, t in enumerate(toks)])
        assert dev.launch_count() > 0 and dev.lazy_stats()["uncached"] == 0
        r.close()
    finally:
        dev.close()
    scale = np.abs(logits["avx2"]).max(axis=1)
    ours = np.abs(logits["gpu"] - logits["avx2"]).max(axis=1) / scale
    band = np.abs(logits["scalar"] - logits["avx2"]).max(axis=1) / scale
    q = lambda a: [float(np.percentile(a, p)) for p in (0, 25, 50, 75, 100)]      # noqa: E731
    print("7B-shaped 8-layer model, 32 positions: |gpu - ref(avx2 order)| / max|logit|   min/25/50/75/max =", ["%.2e" % v for v in q(ours)])
    print("                                       |ref(scalar) - ref(avx2)| / max|logit| min/25/50/75/max =", ["%.2e" % v for v in q(band)])
    assert np.isfinite(logits["gpu"]).all()
    assert np.median(ours) <= 1.0 * np.median(band) * 1.5 and ours.max() <= 1.5 * band.max(), (q(ours), q(band))
    # greedy choice agrees wherever the reference's own two paths agree
    same = logits["scalar"].argmax(1) == logits["avx2"].argmax(1)
    assert (logits["gpu"].argmax(1)[same] == logits["avx2"].argmax(1)[same]).mean() >= 0.9
