// Mock of the C ABI (include/crabml_cuda.h) for the host-logic test of the C++ Llama2Runner replay
// (crabml_b200/csrc/host/llama2_runner.cpp): every entry point the runner uses only RECORDS the call (op name + views) into
// a trace; no CUDA, no arithmetic.  tests/test_host_runner_trace.py builds llama2_runner.cpp against this file and compares
// the trace with the one the Python replay of the reference's forward() (oracle/llama_replay.py, which reproduced the
// reference's golden generations on its trained models) produces on a trace-only tensor class.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/crabml_cuda.h"

struct cc_buf { int refs; int dtype; int64_t nelems; };
struct cc_device { int dummy; };

static std::vector<std::string> g_trace;
static cc_device g_dev;

static std::string V(const cc_view* v) {
    std::string s = "[";
    for (int i = 0; i < v->ndim; i++) s += (i ? "," : "") + std::to_string((long long)v->shape[i]);
    s += "]/[";
    for (int i = 0; i < v->ndim; i++) s += (i ? "," : "") + std::to_string((long long)v->strides[i]);
    s += "]:" + std::to_string(v->buf->dtype);
    return s;
}
static std::string F(float f) { char b[64]; snprintf(b, sizeof b, "%.9g", (double)f); return b; }
static bool contiguous(const cc_view* v) {
    if (v->ndim == 0) return true;
    if (v->strides[v->ndim - 1] != 1) return false;
    int64_t last = 1;
    for (int i = v->ndim - 1; i >= 0; i--) { if (last != v->strides[i]) return false; last *= v->shape[i]; }
    return true;
}
static cc_buf* newbuf(int dtype, int64_t n) { return new cc_buf{1, dtype, n}; }
static int64_t vlen(const cc_view* v) { int64_t n = 1; for (int i = 0; i < v->ndim; i++) n *= v->shape[i]; return n; }

extern "C" {
// ---- test-side helpers --------------------------------------------------------------------------------------------------
CC_API cc_device* mock_device() { return &g_dev; }
CC_API cc_buf* mock_new_buf(int dtype, int64_t nelems) { return newbuf(dtype, nelems); }
CC_API void mock_trace_clear() { g_trace.clear(); }
CC_API int64_t mock_trace_size() { size_t n = 0; for (auto& s : g_trace) n += s.size() + 1; return (int64_t)n; }
CC_API void mock_trace_copy(char* dst) { for (auto& s : g_trace) { memcpy(dst, s.data(), s.size()); dst += s.size(); *dst++ = '\n'; } }

// ---- the ABI surface the runner uses -----------------------------------------------------------------------------------------
CC_API const char* cc_last_error(cc_device*) { return "mock"; }
CC_API int cc_device_flush(cc_device*) { g_trace.push_back("flush"); return CC_OK; }
CC_API void cc_tensor_retain(cc_buf* b) { b->refs++; }
CC_API void cc_tensor_release(cc_buf* b) { if (--b->refs == 0) delete b; }
CC_API int32_t cc_tensor_dtype(const cc_buf* b) { return b->dtype; }
CC_API int64_t cc_tensor_capacity(const cc_buf* b) { return b->nelems; }
CC_API int cc_tensor_alloc(cc_device*, const int64_t* shape, int32_t ndim, int32_t t, cc_buf** out) {
    int64_t n = 1; std::string s = "alloc [";
    for (int i = 0; i < ndim; i++) { n *= shape[i]; s += (i ? "," : "") + std::to_string((long long)shape[i]); }
    g_trace.push_back(s + "]:" + std::to_string(t));
    *out = newbuf(t, n);
    return CC_OK;
}
CC_API int cc_tensor_dup(cc_device*, const cc_view* src, cc_buf** out) { g_trace.push_back("dup " + V(src)); *out = newbuf(CC_F32, vlen(src)); return CC_OK; }
CC_API int cc_tensor_export_f32(cc_device*, const cc_view* src, float* dst, size_t n) {
    g_trace.push_back("export " + V(src) + " n=" + std::to_string(n));
    for (size_t i = 0; i < n; i++) dst[i] = 0.0f;
    return CC_OK;
}
CC_API int cc_copy_rows_from(cc_device*, const cc_view* dst, const cc_view* src, const int64_t* rows, int32_t n_rows) {
    std::string s = "copy_rows_from dst=" + V(dst) + " src=" + V(src) + " rows=[";
    for (int i = 0; i < n_rows; i++) s += (i ? "," : "") + std::to_string((long long)rows[i]);
    g_trace.push_back(s + "]");
    return CC_OK;
}
CC_API int cc_concatenate(cc_device*, const cc_view* self, const cc_view* rhs, int32_t axis) {
    g_trace.push_back("concatenate dst=" + V(self) + " src=" + V(rhs) + " axis=" + std::to_string(axis));
    return CC_OK;
}
CC_API int cc_contiguous(cc_device*, const cc_view* src, cc_buf** out) {
    if (contiguous(src)) { src->buf->refs++; *out = src->buf; return CC_OK; }      // api.rs:40: already contiguous -> same storage
    g_trace.push_back("contiguous " + V(src));
    *out = newbuf(src->buf->dtype, vlen(src));
    return CC_OK;
}
CC_API int cc_rope_inplace(cc_device*, const cc_view* x, int32_t mode, int64_t pos, int64_t dims) {
    g_trace.push_back("rope " + V(x) + " mode=" + std::to_string(mode) + " pos=" + std::to_string((long long)pos) + " dims=" + std::to_string((long long)dims));
    return CC_OK;
}
CC_API int cc_rms_norm_inplace(cc_device*, const cc_view* x, float eps) { g_trace.push_back("rms_norm " + V(x) + " eps=" + F(eps)); return CC_OK; }
CC_API int cc_softmax_inplace(cc_device*, const cc_view* x, int32_t axis) { g_trace.push_back("softmax " + V(x) + " axis=" + std::to_string(axis)); return CC_OK; }
CC_API int cc_silu_inplace(cc_device*, const cc_view* x) { g_trace.push_back("silu " + V(x)); return CC_OK; }
CC_API int cc_gelu_inplace(cc_device*, const cc_view* x) { g_trace.push_back("gelu " + V(x)); return CC_OK; }
CC_API int cc_mul_inplace(cc_device*, const cc_view* x, const cc_view* r) { g_trace.push_back("mul " + V(x) + " rhs=" + V(r)); return CC_OK; }
CC_API int cc_add_inplace(cc_device*, const cc_view* x, const cc_view* r) { g_trace.push_back("add " + V(x) + " rhs=" + V(r)); return CC_OK; }
CC_API int cc_scale_inplace(cc_device*, const cc_view* x, float f) { g_trace.push_back("scale " + V(x) + " f=" + F(f)); return CC_OK; }
CC_API int cc_matmul_vec(cc_device*, const cc_view* w, const cc_view* x, cc_buf** out) {
    g_trace.push_back("matmul_vec w=" + V(w) + " x=" + V(x));
    *out = newbuf(CC_F32, (x->ndim == 1 ? 1 : x->shape[0]) * w->shape[0]);
    return CC_OK;
}
CC_API int cc_batch_matmul(cc_device*, const cc_view* a, const cc_view* b, cc_buf** out) {
    g_trace.push_back("batch_matmul a=" + V(a) + " b=" + V(b));
    *out = newbuf(CC_F32, a->shape[0] * a->shape[1] * b->shape[2]);
    return CC_OK;
}
CC_API int cc_debug_tensor_tap(cc_device*, const char* name, const cc_view*) { g_trace.push_back(std::string("tap ") + name); return CC_OK; }
CC_API int cc_all_reduce_sum_inplace(cc_device*, const cc_view* x) { g_trace.push_back("all_reduce " + V(x)); return CC_OK; }
CC_API int cc_all_gather(cc_device*, const cc_view* dst, const cc_view* src) { g_trace.push_back("all_gather dst=" + V(dst) + " src=" + V(src)); return CC_OK; }
// greedy decoding on the device (ccr_runner_generate_greedy): the mock's "device" always samples token 7
CC_API int cc_copy_rows_from_slot(cc_device*, const cc_view* dst, const cc_view* src, int32_t slot) {
    g_trace.push_back("copy_rows_from_slot dst=" + V(dst) + " src=" + V(src) + " slot=" + std::to_string(slot));
    return CC_OK;
}
CC_API int cc_argmax_to_slot(cc_device*, const cc_view* x, int32_t slot, int64_t hist) {
    g_trace.push_back("argmax_to_slot " + V(x) + " slot=" + std::to_string(slot) + " hist=" + std::to_string((long long)hist));
    return CC_OK;
}
CC_API int cc_read_history(cc_device*, int64_t first, int64_t count, int64_t* out) {
    g_trace.push_back("read_history first=" + std::to_string((long long)first) + " count=" + std::to_string((long long)count));
    for (int64_t i = 0; i < count; i++) out[i] = 7;
    return CC_OK;
}
CC_API int cc_tensor_export_f32_async(cc_device*, const cc_view* src, float* dst, size_t n) {
    g_trace.push_back("export_async " + V(src) + " n=" + std::to_string(n));
    for (size_t i = 0; i < n; i++) dst[i] = 0.0f;
    return CC_OK;
}
CC_API int cc_device_synchronize(cc_device*) { g_trace.push_back("synchronize"); return CC_OK; }
CC_API int cc_host_alloc(cc_device*, size_t bytes, void** out) { *out = malloc(bytes ? bytes : 1); return CC_OK; }
CC_API void cc_host_free(cc_device*, void* p) { free(p); }
}
