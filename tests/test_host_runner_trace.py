"""Host logic of the product's C++ Llama2Runner replay (crabml_b200/csrc/host/llama2_runner.cpp) on CPU: built against a mock
of the C ABI that only records calls, its op trace must equal, call for call (op, shapes, strides, dtypes, scalars, tap names),
the trace of the Python replay of the reference's forward() (oracle/llama_replay.py -- the replay that reproduced the
reference's golden generations on its trained models) run on a trace-only tensor class.  Covers the
single-device order (llama2.rs:184-281, 527-638) and the sharded insertion points (all_reduce after wo / ffn_down,
all_gather of the logits)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from crabml_b200 import capi, sharding
from oracle import oracle as oc
from oracle.llama_replay import Llama2Runner, LlamaConfig as OConf, LlamaWeights
from oracle.tensor_ref import TensorStrider

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _f(x):
    return "%.9g" % float(np.float32(x))


class TraceDevice:
    def __init__(self):
        self.trace = []


class TraceTensor:
    """The Tensor trait with metadata only: every data op appends one line to device.trace (format of tests/host/mock_abi.cpp)."""

    def __init__(self, strider, dtype, device, capacity):
        self._strider, self._dtype, self.device, self.capacity = strider, dtype, device, capacity

    def V(self):
        st = self._strider
        return f"[{','.join(map(str, st.shape))}]/[{','.join(map(str, st.strides))}]:{self._dtype}"

    def log(self, s): self.device.trace.append(s)

    @classmethod
    def weight(cls, shape, dtype, device):
        return cls(TensorStrider(shape), dtype, device, int(np.prod(shape)))

    @classmethod
    def alloc(cls, shape, dtype, device):
        device.trace.append(f"alloc [{','.join(map(str, shape))}]:{dtype}")
        return cls(TensorStrider(shape), dtype, device, int(np.prod(shape)))

    def dtype(self): return self._dtype
    def shape(self): return list(self._strider.shape)
    def strider(self): return self._strider
    def _with(self, st): return TraceTensor(st, self._dtype, self.device, self.capacity)

    def resize(self, axis, n):
        ns = self.shape(); ns[axis] = n
        assert int(np.prod(ns)) <= self.capacity
        return self._with(self._strider.resize(ns))

    def with_strider(self, st): return self._with(st.clone())
    def reshape(self, shape): return self._with(self._strider.reshape(list(shape)))
    def transpose(self, dims): return self._with(self._strider.transpose(list(dims)))
    def with_name(self, name): self.log(f"tap {name}"); return self

    def contiguous(self):
        if self._strider.is_contiguous():
            return self
        self.log(f"contiguous {self.V()}")
        return TraceTensor(TensorStrider(self.shape()), self._dtype, self.device, self._strider.len())

    def concatenate(self, rhs, axis):
        self.log(f"concatenate dst={self.V()} src={rhs.V()} axis={axis}")
        ns = self.shape(); ns[axis] += rhs.shape()[axis]
        self._strider = self._strider.resize(ns)

    def copy_rows_from(self, src, rows): self.log(f"copy_rows_from dst={self.V()} src={src.V()} rows=[{','.join(map(str, rows))}]")
    def export(self): self.log(f"export {self.V()} n={self._strider.len()}"); return np.zeros(self._strider.len(), np.float32)
    def dup(self): self.log(f"dup {self.V()}"); return TraceTensor(TensorStrider(self.shape()), oc.F32, self.device, self._strider.len())
    def rope_inplace(self, mode, pos, dims): self.log(f"rope {self.V()} mode={mode} pos={pos} dims={dims}"); return self
    def rms_norm_inplace(self, eps): self.log(f"rms_norm {self.V()} eps={_f(eps)}"); return self
    def softmax_inplace(self, axis): self.log(f"softmax {self.V()} axis={axis}"); return self
    def silu_inplace(self): self.log(f"silu {self.V()}"); return self
    def gelu_inplace(self): self.log(f"gelu {self.V()}"); return self
    def mul_inplace(self, r): self.log(f"mul {self.V()} rhs={r.V()}"); return self
    def add_inplace(self, r): self.log(f"add {self.V()} rhs={r.V()}"); return self
    def scale_inplace(self, f): self.log(f"scale {self.V()} f={_f(f)}"); return self
    def all_reduce_sum_inplace(self): self.log(f"all_reduce {self.V()}"); return self
    def all_gather_from(self, piece): self.log(f"all_gather dst={self.V()} src={piece.V()}"); return self

    def matmul_vec(self, x):
        self.log(f"matmul_vec w={self.V()} x={x.V()}")
        shape = [self.shape()[0]] if len(x.shape()) == 1 else [x.shape()[0], self.shape()[0]]
        return TraceTensor(TensorStrider(shape), oc.F32, self.device, int(np.prod(shape)))

    def batch_matmul(self, b):
        self.log(f"batch_matmul a={self.V()} b={b.V()}")
        shape = [self.shape()[0], self.shape()[1], b.shape()[2]]
        return TraceTensor(TensorStrider(shape), oc.F32, self.device, int(np.prod(shape)))


@pytest.fixture(scope="module")
def mock_runner(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("mockabi") / "librunner_mock.so")
    srcs = [os.path.join(ROOT, "crabml_b200", "csrc", "host", "llama2_runner.cpp"), os.path.join(ROOT, "tests", "host", "mock_abi.cpp")]
    subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", *srcs, "-o", out], check=True, capture_output=True, timeout=300)
    L = C.CDLL(out)
    L.mock_device.restype = C.c_void_p
    L.mock_new_buf.restype, L.mock_new_buf.argtypes = C.c_void_p, [C.c_int, C.c_int64]
    L.mock_trace_size.restype = C.c_int64
    L.mock_trace_copy.argtypes = [C.c_char_p]
    L.ccr_runner_create.argtypes = [C.c_void_p, C.POINTER(capi.ccr_llama_config), C.POINTER(capi.ccr_llama_weights), C.c_int32, C.POINTER(C.c_void_p)]
    L.ccr_runner_forward.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_int64, C.c_void_p]
    L.ccr_runner_last_error.restype, L.ccr_runner_last_error.argtypes = C.c_char_p, [C.c_void_p]
    L.ccr_runner_destroy.argtypes = [C.c_void_p]
    return L


def _cpp_trace(L, conf, wt, ct, f16_kv, plan, steps, kv_seq):
    world = plan.world if plan else 1
    dim, hd = conf.embedding_dim, conf.embedding_dim // conf.n_heads
    hid = plan.hidden_local if plan else conf.hidden_dim
    qd, kvd, vocab_rows = hd * conf.n_heads // world, hd * conf.n_kv_heads // world, conf.vocab_size // world
    nl = conf.n_layers
    keep = []

    def arr(dtype, n):
        a = (C.c_void_p * nl)(*[L.mock_new_buf(dtype, n) for _ in range(nl)])
        keep.append(a)
        return C.cast(a, C.POINTER(C.c_void_p))
    w = capi.ccr_llama_weights(L.mock_new_buf(wt, conf.vocab_size * dim), arr(wt, qd * dim), arr(wt, kvd * dim), arr(wt, kvd * dim),
                               arr(wt, dim * qd), arr(wt, hid * dim), arr(wt, dim * hid), arr(wt, hid * dim), arr(oc.F32, dim),
                               arr(oc.F32, dim), L.mock_new_buf(oc.F32, dim), L.mock_new_buf(ct, vocab_rows * dim))
    cconf = capi.ccr_llama_config(conf.n_heads, conf.n_kv_heads, nl, dim, conf.hidden_dim, conf.seq_len, conf.vocab_size,
                                  conf.rope_dim or 0, conf.rms_norm_eps, int(f16_kv), plan.rank if plan else 0, world, hid)
    h = C.c_void_p()
    L.mock_trace_clear()
    rc = L.ccr_runner_create(L.mock_device(), C.byref(cconf), C.byref(w), kv_seq, C.byref(h))
    assert rc == 0
    logits = np.zeros(conf.vocab_size, np.float32)
    for pos, tok in steps:
        t = (C.c_int64 * 1)(tok)
        rc = L.ccr_runner_forward(h, t, 1, pos, logits.ctypes.data_as(C.c_void_p))
        assert rc == 0, L.ccr_runner_last_error(h)
    buf = C.create_string_buffer(int(L.mock_trace_size()) + 1)
    L.mock_trace_copy(buf)
    L.ccr_runner_destroy(h)
    return buf.value.decode().splitlines()


def _py_trace(conf, wt, ct, f16_kv, plan, steps, kv_seq):
    dev = TraceDevice()
    world = plan.world if plan else 1
    dim, hd = conf.embedding_dim, conf.embedding_dim // conf.n_heads
    hid = plan.hidden_local if plan else conf.hidden_dim
    qd, kvd, vocab_rows = hd * conf.n_heads // world, hd * conf.n_kv_heads // world, conf.vocab_size // world
    nl = conf.n_layers

    def W(shape, t): return TraceTensor.weight(shape, t, dev)
    lw = LlamaWeights(token_embed=W([conf.vocab_size, dim], wt), wq=[W([qd, dim], wt) for _ in range(nl)], wk=[W([kvd, dim], wt) for _ in range(nl)],
                      wv=[W([kvd, dim], wt) for _ in range(nl)], wo=[W([dim, qd], wt) for _ in range(nl)],
                      ffn_gate_weight=[W([hid, dim], wt) for _ in range(nl)], ffn_down_weight=[W([dim, hid], wt) for _ in range(nl)],
                      ffn_up_weight=[W([hid, dim], wt) for _ in range(nl)], rms_att_weight=[W([dim], oc.F32) for _ in range(nl)],
                      rms_ffn_weight=[W([dim], oc.F32) for _ in range(nl)], rms_final_weight=W([dim], oc.F32), output_weight=W([vocab_rows, dim], ct))
    r = Llama2Runner(TraceTensor, conf, lw, dev, kv_seq, use_f16_kv_cache=f16_kv, world=world)
    for pos, tok in steps:
        r.forward([tok], pos)
    return dev.trace


@pytest.mark.parametrize("name,conf,f16_kv,world", [
    ("tinyllamas", OConf(6, 6, 6, 288, 768, 256, 32000, 1e-5, 48), False, 1),
    ("llama2-7b-shape", OConf(32, 32, 2, 4096, 11008, 4096, 32000, 1e-5, 128), False, 1),
    ("gqa-f16kv", OConf(32, 8, 2, 4096, 14336, 4096, 32000, 1e-5, 128), True, 1),
    ("llama2-7b-sharded-x4", OConf(32, 32, 2, 4096, 11008, 4096, 32000, 1e-5, 128), False, 4),
])
def test_cpp_runner_issues_the_reference_op_sequence(mock_runner, name, conf, f16_kv, world):
    plan = None
    if world > 1:
        plan = sharding.make_plan(conf.n_heads, conf.n_kv_heads, conf.embedding_dim, conf.hidden_dim, conf.vocab_size, oc.Q8_0, 1, world, f16_kv)
    steps = [(0, 1), (1, 365), (2, 2354)]
    got = _cpp_trace(mock_runner, conf, oc.Q8_0, oc.Q8_0, f16_kv, plan, steps, 16)
    want = _py_trace(conf, oc.Q8_0, oc.Q8_0, f16_kv, plan, steps, 16)
    # the KV caches are allocated at construction on both sides; compare everything
    assert len(got) == len(want), (len(got), len(want), [(a, b) for a, b in zip(got, want) if a != b][:5])
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, f"call {i}: C++ runner `{a}` vs reference replay `{b}`"
    per_token = (len(got) - 2 * conf.n_layers) // len(steps)
    assert sum(1 for ln in got if ln.startswith("matmul_vec")) == len(steps) * (7 * conf.n_layers + 1)
    if world > 1:
        assert sum(1 for ln in got if ln.startswith("all_reduce")) == len(steps) * 2 * conf.n_layers
        assert sum(1 for ln in got if ln.startswith("all_gather")) == len(steps)
    assert per_token > 0


def test_cpp_runner_greedy_loop_keeps_the_reference_forward_and_samples_on_the_device(mock_runner):
    """ccr_runner_generate_greedy: the op sequence of every step is the reference's forward() (llama2.rs:184-281) with two
    substitutions only -- the embedding lookup of a generated token reads its id from a device slot, and the sampler's argmax
    (sampler.rs:109-116) runs on the device -- and the step budget follows llama2.rs:141-152 (first token from the prompt pass,
    then min(steps - 1, seq_len - pos - 1) more)."""
    L = mock_runner
    conf = OConf(6, 6, 2, 288, 768, 256, 32000, 1e-5, 48)
    dim, nl = conf.embedding_dim, conf.n_layers
    keep = []

    def arr(dtype, n):
        a = (C.c_void_p * nl)(*[L.mock_new_buf(dtype, n) for _ in range(nl)])
        keep.append(a)
        return C.cast(a, C.POINTER(C.c_void_p))
    wt = oc.Q8_0
    w = capi.ccr_llama_weights(L.mock_new_buf(wt, conf.vocab_size * dim), arr(wt, dim * dim), arr(wt, dim * dim), arr(wt, dim * dim), arr(wt, dim * dim),
                               arr(wt, 768 * dim), arr(wt, dim * 768), arr(wt, 768 * dim), arr(oc.F32, dim), arr(oc.F32, dim), L.mock_new_buf(oc.F32, dim),
                               L.mock_new_buf(wt, conf.vocab_size * dim))
    cconf = capi.ccr_llama_config(6, 6, nl, dim, 768, 256, 32000, 48, 1e-5, 0, 0, 1, 768)
    h = C.c_void_p()
    assert L.ccr_runner_create(L.mock_device(), C.byref(cconf), C.byref(w), 32, C.byref(h)) == 0
    L.ccr_runner_generate_greedy.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    L.mock_trace_clear()
    prompt = (C.c_int64 * 2)(1, 365)
    out = (C.c_int64 * 8)()
    n = C.c_int32(0)
    assert L.ccr_runner_generate_greedy(h, prompt, 2, 4, -1, out, C.byref(n)) == 0, L.ccr_runner_last_error(h)
    buf = C.create_string_buffer(int(L.mock_trace_size()) + 1)
    L.mock_trace_copy(buf)
    got = buf.value.decode().splitlines()
    L.ccr_runner_destroy(h)
    assert n.value == 4 and list(out[:4]) == [7, 7, 7, 7]
    # reference forwards of the same 5 positions: prompt[0], prompt[1], then three generated tokens
    want = _py_trace(conf, wt, wt, False, None, [(0, 1), (1, 365), (2, 0), (3, 0), (4, 0)], 32)[2 * nl:]     # skip the KV-cache allocs
    norm = []
    for ln in got:
        if ln.startswith("copy_rows_from_slot"):
            ln = ln.replace("copy_rows_from_slot", "copy_rows_from").replace(" slot=0", " rows=[0]")
        norm.append(ln)
    body = [ln for ln in norm if not ln.startswith(("argmax_to_slot", "flush", "read_history", "export"))]
    ref = [ln for ln in want if not ln.startswith("export")]
    assert body == ref
    assert [ln for ln in got if ln.startswith("argmax_to_slot")] == [f"argmax_to_slot [32000]/[1]:0 slot=0 hist={i}" for i in range(4)]
    assert got[-1] == "read_history first=0 count=4"
    assert sum(1 for ln in got if ln.startswith("copy_rows_from_slot")) == 3


@pytest.mark.parametrize("arch", ["qwen2", "gemma"])
def test_cpp_runner_other_architectures_issue_the_reference_op_sequence(mock_runner, arch):
    """forward_qwen2 (llama2.rs:283-352: bias adds on q/k/v, Neox RoPE) and forward_gemma (llama2.rs:455-524: embedding scaled by
    sqrt(dim), 2-d q/k views, Neox RoPE, GeLU ffn, tied classifier): the C++ replay against the Python replay, call for call."""
    L = mock_runner
    conf = OConf(8, 4, 2, 256, 512, 64, 1000, 1e-6, 32, arch)
    dim, nl, hd = conf.embedding_dim, conf.n_layers, 32
    qd, kvd = hd * conf.n_heads, hd * conf.n_kv_heads
    wt = oc.Q8_0
    keep = []

    def arr(dtype, n):
        a = (C.c_void_p * nl)(*[L.mock_new_buf(dtype, n) for _ in range(nl)])
        keep.append(a)
        return C.cast(a, C.POINTER(C.c_void_p))
    tied = arch == "gemma"
    w = capi.ccr_llama_weights(L.mock_new_buf(wt, conf.vocab_size * dim), arr(wt, qd * dim), arr(wt, kvd * dim), arr(wt, kvd * dim), arr(wt, dim * qd),
                               arr(wt, 512 * dim), arr(wt, dim * 512), arr(wt, 512 * dim), arr(oc.F32, dim), arr(oc.F32, dim), L.mock_new_buf(oc.F32, dim),
                               None if tied else L.mock_new_buf(wt, conf.vocab_size * dim),
                               arr(oc.F32, qd) if arch == "qwen2" else None, arr(oc.F32, kvd) if arch == "qwen2" else None, arr(oc.F32, kvd) if arch == "qwen2" else None)
    cconf = capi.ccr_llama_config(8, 4, nl, dim, 512, 64, 1000, 32, 1e-6, 0, 0, 1, 512, {"qwen2": 1, "gemma": 2}[arch])
    h = C.c_void_p()
    L.mock_trace_clear()
    assert L.ccr_runner_create(L.mock_device(), C.byref(cconf), C.byref(w), 16, C.byref(h)) == 0, L.ccr_runner_last_error(h)
    logits = np.zeros(conf.vocab_size, np.float32)
    steps = [(0, 1), (1, 365)]
    for pos, tok in steps:
        t = (C.c_int64 * 1)(tok)
        assert L.ccr_runner_forward(h, t, 1, pos, logits.ctypes.data_as(C.c_void_p)) == 0, L.ccr_runner_last_error(h)
    buf = C.create_string_buffer(int(L.mock_trace_size()) + 1)
    L.mock_trace_copy(buf)
    got = buf.value.decode().splitlines()
    L.ccr_runner_destroy(h)
    dev = TraceDevice()

    def W(shape, t): return TraceTensor.weight(shape, t, dev)
    lw = LlamaWeights(token_embed=W([conf.vocab_size, dim], wt), wq=[W([qd, dim], wt) for _ in range(nl)], wk=[W([kvd, dim], wt) for _ in range(nl)],
                      wv=[W([kvd, dim], wt) for _ in range(nl)], wo=[W([dim, qd], wt) for _ in range(nl)],
                      ffn_gate_weight=[W([512, dim], wt) for _ in range(nl)], ffn_down_weight=[W([dim, 512], wt) for _ in range(nl)],
                      ffn_up_weight=[W([512, dim], wt) for _ in range(nl)], rms_att_weight=[W([dim], oc.F32) for _ in range(nl)],
                      rms_ffn_weight=[W([dim], oc.F32) for _ in range(nl)], rms_final_weight=W([dim], oc.F32),
                      output_weight=None if tied else W([conf.vocab_size, dim], wt),
                      bq=[W([qd], oc.F32) for _ in range(nl)], bk=[W([kvd], oc.F32) for _ in range(nl)], bv=[W([kvd], oc.F32) for _ in range(nl)])
    r = Llama2Runner(TraceTensor, conf, lw, dev, 16)
    for pos, tok in steps:
        r.forward([tok], pos)
    want = dev.trace
    assert len(got) == len(want), (len(got), len(want), [(a, b) for a, b in zip(got, want) if a != b][:5])
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, f"{arch} call {i}: C++ runner `{a}` vs reference replay `{b}`"
    assert any(ln.startswith("rope") and "mode=1" in ln for ln in got)
    if arch == "gemma":
        assert any(ln.startswith("gelu") for ln in got) and any(ln.startswith("scale") for ln in got) and any(ln.startswith("tap scaled_embed") for ln in got)
    else:
        assert sum(1 for ln in got if ln.startswith("add") and ":0 rhs=[256]" in ln or ln.startswith("add") and "rhs=[128]" in ln) >= 2 * nl
