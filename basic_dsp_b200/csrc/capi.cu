// C ABI of basic_dsp_b200 (include/basic_dsp_b200.h): device-resident vector handles behind the
// reference's interop function names (interop/src/facade32.rs / facade64.rs), plus the batched
// raw-pointer kernels.  Host logic only; all arithmetic runs in the CUDA kernels of this directory.
#include <math.h>
#include <string.h>

#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <vector>

#include "../../include/basic_dsp_b200.h"
#include "common.cuh"
#include "conv.cuh"
#include "elementwise.cuh"
#include "mathops.cuh"
#include "fft.cuh"
#include "interp.cuh"

using namespace bdsp;

namespace {

thread_local cudaStream_t g_stream = 0;

enum {
    E_OK = 0, E_INVALID = -1, E_SAME_SIZE = 1, E_META = 2, E_COMPLEX = 3, E_REAL = 4, E_TIME = 5, E_FREQ = 6,
    E_ARG_LEN = 7, E_EVEN_LEN = 13, E_RESIZE = 14, VOID_OK = 9
};

// InteropVec<T> analogue: device storage + device scratch ("SingleBuffer": never shrinks, results are
// produced in the scratch and swapped in = `trade`, vector/src/vector_types/support_std.rs:79-81)
template <typename T> struct Vec {
    T* d = nullptr;        size_t cap = 0;    // storage, capacity in T scalars
    T* scratch = nullptr;  size_t scap = 0;
    size_t len = 0;                           // valid_len in T scalars
    T delta = 1;
    int is_complex = 0;
    int domain = 0;                           // 0 time, 1 frequency
    unsigned long long version = 0;           // bumped by every mutation (invalidates caches)
    // cache: overlap-save plan of this vector used as impulse response.  The vector is only BORROWED by
    // convolve_signal (`&VecBuf`, facade32.rs:1171), possibly by several threads at once: the cache is guarded by
    // `plan_mu`, and the plan is immutable and reference counted (a caller keeps it alive while its kernel is queued).
    std::mutex plan_mu;
    std::shared_ptr<OlsPlan> plan; unsigned long long plan_version = ~0ull; int plan_complex_signal = -1;
    // host mirror for data32()
    std::vector<T> host;
};

template <typename T> struct Res { int32_t result_code; Vec<T>* vector; };

template <typename T> bool erroneous(const Vec<T>* v) { return v->len == 0 && isnan((double)v->delta); }
template <typename T> void mark_invalid(Vec<T>* v) { v->len = 0; v->delta = (T)NAN; v->version++; }
template <typename T> Res<T> done(Vec<T>* v, int code) {
    v->version++;
    Res<T> r;
    r.result_code = code != 0 ? code : (erroneous(v) ? E_INVALID : E_OK);
    r.vector = v;
    return r;
}
template <typename T> size_t points_of(const Vec<T>* v) { return v->is_complex ? v->len / 2 : v->len; }

template <typename T> int reserve(T** p, size_t* cap, size_t want, bool keep, size_t keep_n) {
    if (*cap >= want) return 0;
    T* n = nullptr;
    BDSP_CUDA_OK(cudaMalloc(&n, (want ? want : 1) * sizeof(T)));
    if (keep && *p && keep_n) BDSP_CUDA_OK(cudaMemcpyAsync(n, *p, keep_n * sizeof(T), cudaMemcpyDeviceToDevice, g_stream));
    if (*p) {
        BDSP_CUDA_OK(cudaStreamSynchronize(g_stream));
        BDSP_CUDA_OK(cudaFree(*p));
    }
    *p = n;
    *cap = want;
    return 0;
}
template <typename T> int ensure_scratch(Vec<T>* v, size_t n) { return reserve(&v->scratch, &v->scap, n, false, 0); }
template <typename T> void trade(Vec<T>* v) {
    T* p = v->d; v->d = v->scratch; v->scratch = p;
    size_t c = v->cap; v->cap = v->scap; v->scap = c;
}

template <typename T> Vec<T>* vec_new(int is_complex, int domain, T init, size_t length, T delta) {
    Vec<T>* v = new Vec<T>();
    v->is_complex = is_complex != 0;
    v->domain = domain == 0 ? 0 : 1;
    v->delta = delta;
    // allocation failure: null handle (bdsp_last_error() says why) instead of taking the host process down
    if (reserve(&v->d, &v->cap, length, false, 0) != 0) { delete v; return nullptr; }
    // to_gen_dsp_vec: a complex vector needs an even number of scalars (support_std.rs:369)
    v->len = (v->is_complex && (length % 2)) ? 0 : length;
    if (length) ew_fill<T>(v->d, length, (double)init, g_stream);
    return v;
}

template <typename T> void vec_delete(Vec<T>* v) {
    if (!v) return;
    cudaStreamSynchronize(g_stream);
    if (v->d) cudaFree(v->d);
    if (v->scratch) cudaFree(v->scratch);
    v->plan.reset();
    delete v;
}

template <typename T> int vec_resize(Vec<T>* v, size_t len) {
    if (v->is_complex && (len % 2)) return E_EVEN_LEN;
    if (len > v->cap) {
        size_t old = v->cap;
        int rc = reserve(&v->d, &v->cap, len, true, old);
        if (rc) return rc;
        // Vec::resize(len, 0): new storage is zero filled (support_std.rs:227-230)
        BDSP_CUDA_OK(cudaMemsetAsync(v->d + old, 0, (len - old) * sizeof(T), g_stream));
    }
    v->len = len;
    v->version++;
    return 0;
}

template <typename T> bool meta_agrees(const Vec<T>* a, const Vec<T>* b) {
    // assert_meta_data! (elementary.rs:370-381, convolution.rs:257-268)
    T ratio = a->delta / b->delta;
    return a->is_complex == b->is_complex && a->domain == b->domain && !(ratio > (T)1.1) && !(ratio < (T)0.9);
}

// ---- transforms ------------------------------------------------------------------------------------
// built-in windows: 0 triangular, 1 hamming, 2 blackman-harris; any other kind is rectangular (interop/src/lib.rs:153-164)
const int RECTANGULAR = 3;

// Options of a transform of `points` points.  shift: fft_shift on the store of a forward transform (freq.rs:85-87), or
// scale(1/points) -> ifft_shift on the load of an inverse one; a built-in window rides on the load.
template <typename T> FftOpts fft_opts(size_t points, bool inverse, bool shift, bool magnitude, bool real_input, int window) {
    FftOpts o;
    o.inverse = inverse;
    o.real_input = real_input;
    o.magnitude = magnitude;
    if (shift && points) {
        if (inverse) { o.in_rot = points / 2; o.scale = (double)((T)1 / (T)points); }
        else o.out_rot = points / 2;
    }
    if (window >= 0 && window < RECTANGULAR) { o.in_mul.kind = 3; o.in_mul.arg = window; }
    return o;
}

// window_table: a host-built window table multiplied in on the load, instead of a built-in window
template <typename T>
Res<T> op_fft(Vec<T>* v, bool inverse, bool shifted, bool magnitude, int window = RECTANGULAR, const T* window_table = nullptr) {
    // time_to_freq.rs:136-165, freq_to_time.rs:138-168, time_freq/mod.rs:32-63
    const int want_domain = inverse ? 1 : 0;
    if (v->domain != want_domain) {
        mark_invalid(v);
        v->is_complex = 1;
        v->domain = 1;
        return done(v, 0);
    }
    const size_t points = points_of(v);
    FftOpts o = fft_opts<T>(points, inverse, shifted, magnitude, !v->is_complex, window);
    if (window_table) { o.in_mul.p = window_table; o.in_mul.kind = 1; }
    if (points) {
        const size_t out_scalars = magnitude ? points : 2 * points;
        int rc = ensure_scratch(v, 2 * points);
        if (!rc) rc = fft_exec<T>(v->d, v->scratch, points, 1, o, nullptr, 0, g_stream);
        if (rc) return done(v, rc);
        trade(v);
        v->len = out_scalars;
    }
    v->delta = (T)points * v->delta;                                           // Q1: both directions
    v->is_complex = magnitude ? 0 : 1;
    v->domain = inverse ? 0 : 1;                                               // Q2: ifft reports Time
    return done(v, 0);
}

template <typename T> Res<T> op_rotate(Vec<T>* v, bool forward) {
    // swap_halves_priv (vector_types/mod.rs:510-524): new[(p + step) % n] = old[p]
    const size_t n = points_of(v);
    if (n < 2) return done(v, 0);
    const size_t step = forward ? n / 2 : n - n / 2;
    int rc = ensure_scratch(v, v->len);
    if (!rc) rc = ew_rotate<T>(v->d, v->scratch, n, step, v->is_complex ? 2 : 1, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    return done(v, 0);
}

template <typename T> Res<T> op_zero_interleave(Vec<T>* v, int factor) {
    if (factor < 1) return done(v, E_ARG_LEN);
    const size_t n = points_of(v);
    const size_t new_len = v->len * (size_t)factor;
    if (n) {
        int rc = ensure_scratch(v, new_len);
        if (!rc) rc = ew_zero_interleave<T>(v->d, v->scratch, n, factor, v->is_complex ? 2 : 1, g_stream);
        if (rc) return done(v, rc);
        trade(v);
    }
    v->len = new_len;
    return done(v, 0);
}

template <typename T> Res<T> op_to_complex(Vec<T>* v) {
    // to_complex_b (real_to_complex.rs:96-111)
    if (v->is_complex) { mark_invalid(v); return done(v, 0); }
    Res<T> r = op_zero_interleave(v, 2);
    v->is_complex = 1;
    return done(v, r.result_code);
}

template <typename T> Res<T> op_zero_pad(Vec<T>* v, size_t points, int option) {
    // zero_pad_b (data_reorganization.rs:407-463)
    const size_t len_before = v->len;
    const size_t step = v->is_complex ? 2 : 1;
    const size_t len = step * points;
    if (len <= len_before) return done(v, E_ARG_LEN);
    int rc = ensure_scratch(v, len);
    if (rc) return done(v, rc);
    T* t = v->scratch;
    cudaMemsetAsync(t, 0, len * sizeof(T), g_stream);
    if (option == 0) {
        cudaMemcpyAsync(t, v->d, len_before * sizeof(T), cudaMemcpyDeviceToDevice, g_stream);
    } else if (option == 1) {
        size_t diff = (len - len_before) / step;
        size_t right = diff / 2, left = (diff - right) * step;
        cudaMemcpyAsync(t + left, v->d, len_before * sizeof(T), cudaMemcpyDeviceToDevice, g_stream);
    } else {
        size_t pb = len_before / step;
        size_t right = (pb / 2) * step, left = (pb - pb / 2) * step;
        cudaMemcpyAsync(t + len - right, v->d + len_before - right, right * sizeof(T), cudaMemcpyDeviceToDevice, g_stream);
        cudaMemcpyAsync(t, v->d, left * sizeof(T), cudaMemcpyDeviceToDevice, g_stream);
    }
    trade(v);
    v->len = len;
    return done(v, 0);
}

// ---- elementwise -----------------------------------------------------------------------------------
template <typename T> Res<T> op_binary(Vec<T>* v, const Vec<T>* o, int op) {
    // elementary.rs:383-455,540-589
    if (v->len != o->len) return done(v, E_SAME_SIZE);
    if (!meta_agrees(v, o)) return done(v, E_META);
    int rc = 0;
    if (v->len) rc = ew_binary<T>(op, v->d, o->d, v->d, v->len, v->is_complex, g_stream);
    return done(v, rc);
}

template <typename T> Res<T> op_real_const(Vec<T>* v, int op, T c) {
    int rc = 0;
    if (v->len) {
        if (op == EW_OFFSET && v->is_complex) rc = ew_complex_const<T>(EW_OFFSET, v->d, v->d, v->len / 2, (double)c, 0.0, g_stream);
        else rc = ew_scalar<T>(op, v->d, v->d, v->len, (double)c, g_stream);
    }
    return done(v, rc);
}

template <typename T> Res<T> op_complex_const(Vec<T>* v, int op, T re, T im) {
    if (!v->is_complex) { mark_invalid(v); return done(v, 0); }   // assert_complex!
    int rc = 0;
    if (v->len) rc = ew_complex_const<T>(op, v->d, v->d, v->len / 2, (double)re, (double)im, g_stream);
    return done(v, rc);
}

template <typename T> Res<T> op_complex_divide(Vec<T>* v, T re, T im) {
    // Complex::new(1,0) / Complex::new(re,im) evaluated in T (num-complex Div), facade32.rs:550-557
    T ns = re * re + im * im;
    T qr = ((T)1 * re + (T)0 * im) / ns;
    T qi = ((T)0 * re - (T)1 * im) / ns;
    return op_complex_const(v, EW_SCALE, qr, qi);
}

template <typename T> Res<T> op_c2r(Vec<T>* v, int op) {
    // complex_to_real.rs:365-478
    if (!v->is_complex) { mark_invalid(v); v->is_complex = 0; return done(v, 0); }
    const size_t points = v->len / 2;
    if (points) {
        int rc = ensure_scratch(v, points);
        if (!rc) rc = ew_complex_to_real<T>(op, v->d, v->scratch, points, g_stream);
        if (rc) return done(v, rc);
        trade(v);
    }
    v->len = points;
    v->is_complex = 0;
    return done(v, 0);
}

template <typename T> int32_t op_get_c2r(Vec<T>* v, Vec<T>* dst, int op) {
    // complex_to_real.rs:595-680; convert_void -> 9 (Q8)
    if (!v->is_complex || dst->is_complex) { dst->len = 0; dst->version++; return VOID_OK; }
    const size_t points = v->len / 2;
    if (vec_resize(dst, points) > 0) return VOID_OK;
    dst->delta = v->delta;
    if (points) {
        int rc = ew_complex_to_real<T>(op, v->d, dst->d, points, g_stream);
        if (rc) return rc;
    }
    dst->version++;
    return VOID_OK;
}

template <typename T> int32_t op_get_mag_phase(Vec<T>* v, Vec<T>* mag, Vec<T>* ph) {
    if (!v->is_complex || mag->is_complex || ph->is_complex) {
        mag->len = 0; ph->len = 0; mag->version++; ph->version++;
        return VOID_OK;
    }
    const size_t points = v->len / 2;
    vec_resize(mag, points);
    vec_resize(ph, points);
    if (points) {
        int rc = ew_mag_phase<T>(v->d, mag->d, ph->d, points, g_stream);
        if (rc) return rc;
    }
    return VOID_OK;
}

// ---- impulse responses evaluated on the host in precision T (conv_types.rs:391-518) ---------------
template <typename T> T host_sinc(T x) {
    if (x == (T)0) return (T)1;
    T pi_x = (T)M_PI * x;
    return (T)sin(pi_x) / pi_x;
}
template <typename T> T host_rc(T x, T rolloff) {
    if (x == (T)0) return (T)1;
    const T one = 1, two = 2, pi = (T)M_PI;
    const T four = two * two;
    if ((T)fabs(x) == one / (two * rolloff)) {
        T arg = pi / two / rolloff;
        return (T)sin(arg) / arg * pi / four;
    }
    T pi_x = pi * x;
    T arg = two * rolloff * x;
    return (T)sin(pi_x) * (T)cos(pi_x * rolloff) / pi_x / (one - (arg * arg));
}

// A real impulse or frequency response: the built-in `kind` (0 sinc, 1 raised cosine with `rolloff`) when `fn` is null,
// else the C callback fn(data, x).  Built-in frequency responses are evaluated on the device, so the host evaluates only
// callbacks and the built-in impulse responses of tap tables.
template <typename T> struct RealFn {
    int kind = 0;
    T rolloff = 0;
    T (*fn)(const void*, T) = nullptr;
    const void* data = nullptr;
    T operator()(T x) const { return fn ? fn(data, x) : kind == 0 ? host_sinc<T>(x) : host_rc<T>(x, rolloff); }
};

// Small host-built tables go through a grow-only pinned staging buffer + device buffer per host thread and device, so
// that a call does no cudaMalloc/cudaFree and never blocks on the GPU: the copy is queued on the caller's stream, the
// consumer kernel follows on the same stream.
struct TableStage {
    void* dev = nullptr;
    void* host = nullptr;
    size_t bytes = 0;
    cudaEvent_t copied = nullptr;   // staging buffer has been read by the last copy
    cudaEvent_t used = nullptr;     // device buffer has been consumed by the last kernel
};
thread_local std::map<int, TableStage> g_stage;   // by device

template <typename T> int stage_table(int dev, const std::vector<T>& h, TableStage** stage) {
    TableStage& s = g_stage[dev];
    const size_t need = (h.size() ? h.size() : 1) * sizeof(T);
    if (!s.copied) {
        BDSP_CUDA_OK(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
        BDSP_CUDA_OK(cudaEventCreateWithFlags(&s.used, cudaEventDisableTiming));
    }
    if (need > s.bytes) {
        BDSP_CUDA_OK(cudaDeviceSynchronize());
        if (s.dev) cudaFree(s.dev);
        if (s.host) cudaFreeHost(s.host);
        s.bytes = need * 2 < 65536 ? 65536 : need * 2;
        BDSP_CUDA_OK(cudaMalloc(&s.dev, s.bytes));
        BDSP_CUDA_OK(cudaMallocHost(&s.host, s.bytes));
    } else {
        BDSP_CUDA_OK(cudaEventSynchronize(s.copied));            // host staging free again (old, tiny copy)
        BDSP_CUDA_OK(cudaStreamWaitEvent(g_stream, s.used, 0));  // device table free again (GPU-side wait)
    }
    memcpy(s.host, h.data(), h.size() * sizeof(T));
    BDSP_CUDA_OK(cudaMemcpyAsync(s.dev, s.host, h.size() * sizeof(T), cudaMemcpyHostToDevice, g_stream));
    BDSP_CUDA_OK(cudaEventRecord(s.copied, g_stream));
    *stage = &s;
    return 0;
}

// ---- cache of tap tables built from the BUILT-IN functions -----------------------------------------------------------
// Repeated calls with the same parameters (the usual streaming use) skip the host evaluation and the upload.
// Keyed by everything the table depends on; tables live in device memory until the process ends (<= 64 entries
// per process, then the cache stops growing).  Callback functions are never cached.
struct TableKey {
    int dev, is64, what, kind, flag;
    double rolloff, a, b;
    size_t n0, n1;
    bool operator<(const TableKey& o) const {
        if (dev != o.dev) return dev < o.dev;
        if (is64 != o.is64) return is64 < o.is64;
        if (what != o.what) return what < o.what;
        if (kind != o.kind) return kind < o.kind;
        if (flag != o.flag) return flag < o.flag;
        if (rolloff != o.rolloff) return rolloff < o.rolloff;
        if (a != o.a) return a < o.a;
        if (b != o.b) return b < o.b;
        if (n0 != o.n0) return n0 < o.n0;
        return n1 < o.n1;
    }
};
std::mutex g_table_mu;
std::map<TableKey, std::pair<void*, size_t>> g_table_cache;

// the key of a table of `f`: built-in functions are cached by parameter set, callbacks are not (nullptr)
template <typename T> const TableKey* cache_key(const RealFn<T>& f, TableKey* key) {
    if (f.fn) return nullptr;
    key->kind = f.kind;
    key->rolloff = (double)f.rolloff;
    return key;
}

// A host-built table on the device for the kernels launched while this object is in scope.  With a key, the table is
// taken from or added to the cache; otherwise, or when the cache is full, build() is staged, and the staging buffer is
// marked consumed when this object goes out of scope, i.e. after the consuming launch.
template <typename T> class DeviceTable {
  public:
    const T* p = nullptr;
    size_t count = 0;   // T scalars
    int rc = 0;
    template <typename Build> DeviceTable(const TableKey* key, Build build) {
        int dev = 0;
        cudaGetDevice(&dev);
        TableKey k = {};
        if (key) {
            k = *key;
            k.dev = dev;
            k.is64 = sizeof(T) == 8;
            std::lock_guard<std::mutex> lk(g_table_mu);
            auto it = g_table_cache.find(k);
            if (it != g_table_cache.end()) {
                p = reinterpret_cast<const T*>(it->second.first);
                count = it->second.second;
                return;
            }
        }
        const std::vector<T> tab = build();
        count = tab.size();
        if (key && cache_insert(k, tab)) return;
        rc = stage_table(dev, tab, &stage_);
        if (!rc) p = reinterpret_cast<const T*>(stage_->dev);
    }
    ~DeviceTable() { if (stage_) cudaEventRecord(stage_->used, g_stream); }
    DeviceTable(const DeviceTable&) = delete;
    DeviceTable& operator=(const DeviceTable&) = delete;

  private:
    TableStage* stage_ = nullptr;
    bool cache_insert(const TableKey& k, const std::vector<T>& tab) {
        std::lock_guard<std::mutex> lk(g_table_mu);
        if (g_table_cache.size() >= 64) return false;
        void* dev = nullptr;
        if (cudaMalloc(&dev, tab.size() * sizeof(T)) != cudaSuccess) return false;
        if (cudaMemcpy(dev, tab.data(), tab.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(dev); return false; }
        g_table_cache[k] = std::make_pair(dev, tab.size());
        p = reinterpret_cast<const T*>(dev);
        return true;
    }
};

// ---- convolution -----------------------------------------------------------------------------------
// convolution with taps resident on the device; h: the impulse-response vector that caches the overlap-save plan of
// these taps between calls, or nullptr (the plan is then made for this call only)
inline std::shared_ptr<OlsPlan> own_plan(OlsPlan* p) { return std::shared_ptr<OlsPlan>(p, [](OlsPlan* q) { ols_plan_destroy(q); }); }

template <typename T>
int convolve_taps(Vec<T>* v, const T* h_dev, size_t L, bool h_complex, Vec<T>* h) {
    const size_t N = points_of(v);
    int rc = ensure_scratch(v, v->len);
    if (rc) return rc;
    std::shared_ptr<OlsPlan> plan;
    if (conv_needs_plan<T>(L, !h_complex)) {
        if (h) {
            std::lock_guard<std::mutex> lk(h->plan_mu);
            if (h->plan && h->plan_version == h->version && h->plan_complex_signal == v->is_complex)
                plan = h->plan;
            else {
                plan = own_plan(ols_plan_create<T>(h_dev, L, !h_complex, v->is_complex != 0, g_stream));
                if (!plan) return -1;
                // other streams may use the plan as soon as it is published
                BDSP_CUDA_OK(cudaStreamSynchronize(g_stream));
                h->plan = plan; h->plan_version = h->version; h->plan_complex_signal = v->is_complex;
            }
        } else {
            plan = own_plan(ols_plan_create<T>(h_dev, L, !h_complex, v->is_complex != 0, g_stream));
            if (!plan) return -1;
        }
    }
    rc = convolve<T>(v->d, v->scratch, N, 1, !v->is_complex, h_dev, L, !h_complex, plan.get(), g_stream);
    // an uncached plan is destroyed here (ols_plan_destroy synchronises the device first)
    if (rc) return rc;
    trade(v);
    return 0;
}

template <typename T> Res<T> op_convolve_signal(Vec<T>* v, Vec<T>* h) {
    // convolution.rs:477-542
    if (!meta_agrees(v, h)) return done(v, E_META);
    if (v->domain != 0) return done(v, E_TIME);
    const size_t N = points_of(v), L = points_of(h);
    if (N < L) return done(v, E_ARG_LEN);
    if (N == 0 || L == 0) {
        if (N) cudaMemsetAsync(v->d, 0, v->len * sizeof(T), g_stream);
        return done(v, 0);
    }
    return done(v, convolve_taps<T>(v, h->d, L, h->is_complex, h));
}

// More taps than points: the tap window wraps around the vector (the reference's ReverseWrappingIterator,
// time_freq/mod.rs:788-848).  Folds Lt taps of `width` scalars each into an N-tap kernel with the same circular result:
// y[i] = sum_k x[(i + cl - 1 - k) mod N] t[k], cl = Lt - Lt/2, re-centred on cl' = N - N/2.
template <typename T> void fold_taps(std::vector<T>& taps, size_t N, size_t width) {
    const size_t Lt = taps.size() / width;
    if (Lt <= N) return;
    std::vector<T> folded(N * width, (T)0);
    const size_t cl = Lt - Lt / 2, cl2 = N - N / 2;
    for (size_t k = 0; k < Lt; k++) {
        const long long off = (long long)cl - 1 - (long long)k;       // x index offset of tap k
        long long k2 = ((long long)cl2 - 1 - off) % (long long)N;     // slot of the N-tap kernel with the same offset
        if (k2 < 0) k2 += (long long)N;
        for (size_t c = 0; c < width; c++) folded[(size_t)k2 * width + c] += taps[k * width + c];
    }
    taps.swap(folded);
}

// convolve_function_priv taps (time_freq/mod.rs:174-213): y[i] = sum_{m=-L..L} x[i+m] f(-m*ratio) == circular FIR with
// h[k] = f(-(L-k)*ratio), k = 0..2L (centre cl = L+1); eval(x, out) writes the `width` scalars of f(x)
template <typename T, typename Eval> std::vector<T> priv_taps(size_t L, T ratio, int width, Eval eval) {
    std::vector<T> h(width * (2 * L + 1));
    T j = -(T)L;
    for (size_t q = 0; q < 2 * L + 1; q++) { eval(-j * ratio, &h[width * (2 * L - q)]); j = j + (T)1; }
    return h;
}

// ratio * f(j/mx * ratio) on the grid j = -mx..: multiply_function_priv with is_fft_shifted = false
// (time_freq/mod.rs:612-723); eval(x, out) writes the `width` scalars of f(x)
template <typename T, typename Eval> std::vector<T> freq_resp_table(size_t points, T ratio, int width, Eval eval) {
    std::vector<T> tab(width * points);
    const size_t offset = points % 2;
    const T mx = (T)(points - offset) / (T)2;
    T j = -(T)(points - offset) / (T)2;
    for (size_t i = 0; i < points; i++) {
        T* t = &tab[width * i];
        eval(j / mx * ratio, t);
        for (int c = 0; c < width; c++) t[c] = ratio * t[c];
        j = j + (T)1;
    }
    return tab;
}

template <typename T, typename CT> auto complex_eval(CT (*fn)(const void*, T), const void* data) {
    return [=](T x, T* out) { const CT c = fn(data, x); out[0] = c.re; out[1] = c.im; };
}

template <typename T> Res<T> op_convolve_fn(Vec<T>* v, const RealFn<T>& f, T ratio, size_t len) {
    // convolution.rs:136-192 (real impulse response)
    if (v->domain != 0) { mark_invalid(v); return done(v, 0); }   // assert_time!
    const size_t N = points_of(v);
    if (N == 0) return done(v, 0);
    const T ratio_inv = (T)1 / ratio;
    const bool simd_branch = len <= 202 && v->len > 2000 && (T)fabs((T)round(ratio_inv) - ratio_inv) < (T)1e-6 && ratio > (T)0.5;
    TableKey key = {};
    key.what = 1; key.flag = simd_branch; key.a = (double)ratio; key.n0 = len; key.n1 = N;
    DeviceTable<T> taps(cache_key(f, &key), [&] {
        std::vector<T> h;
        if (simd_branch) {
            // taps f(j/ratio), j = -len..len, handed to convolve_signal (convolution.rs:151-172).
            // Deviation Q4: for real vectors the reference fills only every second tap.
            T j = -(T)len;
            for (size_t q = 0; q < 2 * len + 1; q++) { h.push_back(f(j * ratio_inv)); j = j + (T)1; }
        } else {
            h = priv_taps<T>(len > N ? N : len, ratio, 1, [&](T x, T* out) { *out = f(x); });
        }
        fold_taps(h, N, 1);
        return h;
    });
    if (taps.rc) return done(v, taps.rc);
    return done(v, convolve_taps<T>(v, taps.p, taps.count, false, nullptr));
}

template <typename T, typename CT>
Res<T> op_convolve_cfn(Vec<T>* v, CT (*fn)(const void*, T), const void* data, T ratio, size_t len) {
    // convolution.rs:195-255 (complex impulse response); only the convolve_function_priv branch of
    // the reference is meaningful (Q5), which is what is implemented for every ratio
    if (!v->is_complex) { mark_invalid(v); return done(v, 0); }
    if (v->domain != 0) { mark_invalid(v); return done(v, 0); }
    const size_t N = points_of(v);
    if (N == 0) return done(v, 0);
    DeviceTable<T> taps(nullptr, [&] {
        std::vector<T> h = priv_taps<T>(len > N ? N : len, ratio, 2, complex_eval<T, CT>(fn, data));
        fold_taps(h, N, 2);   // 2L + 1 > N: the window wraps around the vector, as in the reference
        return h;
    });
    if (taps.rc) return done(v, taps.rc);
    return done(v, convolve_taps<T>(v, taps.p, taps.count / 2, true, nullptr));
}

template <typename T> Res<T> op_mul_freq_resp(Vec<T>* v, const RealFn<T>& f, T ratio) {
    // convolution.rs:576-610 + multiply_function_priv (time_freq/mod.rs:612-723)
    if (v->domain != 1) { mark_invalid(v); return done(v, 0); }
    const size_t points = points_of(v);
    if (!points) return done(v, 0);
    if (!f.fn) return done(v, ew_mul_freq_resp<T>(v->d, points, v->is_complex, f.kind, (double)f.rolloff, (double)ratio, g_stream));
    DeviceTable<T> tab(nullptr, [&] { return freq_resp_table<T>(points, ratio, 1, [&](T x, T* out) { *out = f(x); }); });
    if (tab.rc) return done(v, tab.rc);
    return done(v, ew_mul_table<T>(v->d, tab.p, points, v->is_complex, 0, g_stream));
}

template <typename T, typename CT>
Res<T> op_mul_freq_resp_c(Vec<T>* v, CT (*fn)(const void*, T), const void* data, T ratio) {
    if (!v->is_complex || v->domain != 1) { mark_invalid(v); return done(v, 0); }
    const size_t points = points_of(v);
    if (!points) return done(v, 0);
    DeviceTable<T> tab(nullptr, [&] { return freq_resp_table<T>(points, ratio, 2, complex_eval<T, CT>(fn, data)); });
    if (tab.rc) return done(v, tab.rc);
    return done(v, ew_mul_table<T>(v->d, tab.p, points, 1, 1, g_stream));
}

// ---- SURVEY 8(f) rows: windows, correlation, reverse, decimatei --------------------------------------
// built-in window kind (evaluated on the device), or a foreign callback window fn(data, i, points) (facade32.rs:1030-1044)
template <typename T> struct WinFn {
    int kind = RECTANGULAR;
    T (*fn)(const void*, size_t, size_t) = nullptr;
    const void* data = nullptr;
    bool symmetric = true;
};

// table of a callback window (multiply_window_priv, vector_types/mod.rs:528-598): symmetric windows evaluate the first half
// and mirror it; unapply multiplies by the reciprocal
template <typename T> std::vector<T> window_table(const WinFn<T>& w, size_t points, bool unapply) {
    std::vector<T> tab(points);
    for (size_t i = 0; i < points; i++) {
        const size_t j = !w.symmetric || i < (points + 1) / 2 ? i : points - 1 - i;
        const T x = w.fn(w.data, j, points);
        tab[i] = unapply ? (T)1 / x : x;
    }
    return tab;
}

template <typename T> Res<T> op_window_fn(Vec<T>* v, const WinFn<T>& w, bool unapply) {
    // time.rs:33-66
    if (v->domain != 0) { mark_invalid(v); return done(v, 0); }
    const size_t points = points_of(v);
    if (!points) return done(v, 0);
    if (!w.fn) return done(v, ew_window<T>(v->d, points, v->is_complex, w.kind < 0 || w.kind > 2 ? RECTANGULAR : w.kind, unapply, g_stream));
    DeviceTable<T> tab(nullptr, [&] { return window_table<T>(w, points, unapply); });
    if (tab.rc) return done(v, tab.rc);
    return done(v, ew_mul_table<T>(v->d, tab.p, points, v->is_complex, 0, g_stream));
}
template <typename T> Res<T> op_window(Vec<T>* v, int kind, bool unapply) {
    WinFn<T> w; w.kind = kind;
    return op_window_fn(v, w, unapply);
}

template <typename T> Res<T> op_windowed_fft_fn(Vec<T>* v, const WinFn<T>& w) {
    // time_to_freq.rs:167-175: apply_window, then fft.  The window rides on the first load of the transform
    // (FftOpts::in_mul) instead of making its own pass over the vector: built-in windows are evaluated on the fly,
    // callback windows come from the host-built table.
    if (v->domain != 0) { mark_invalid(v); return op_fft(v, false, true, false); }
    const size_t points = points_of(v);
    if (!points || !w.fn) return op_fft(v, false, true, false, w.kind);
    DeviceTable<T> tab(nullptr, [&] { return window_table<T>(w, points, false); });
    if (tab.rc) return done(v, tab.rc);
    return op_fft(v, false, true, false, RECTANGULAR, tab.p);
}
template <typename T> Res<T> op_windowed_ifft_fn(Vec<T>* v, const WinFn<T>& w) {
    Res<T> r = op_fft(v, true, true, false);
    if (r.result_code) return r;
    return op_window_fn(v, w, true);
}
template <typename T> Res<T> op_windowed_fft(Vec<T>* v, int kind) { WinFn<T> w; w.kind = kind; return op_windowed_fft_fn(v, w); }
template <typename T> Res<T> op_windowed_ifft(Vec<T>* v, int kind) { WinFn<T> w; w.kind = kind; return op_windowed_ifft_fn(v, w); }

template <typename T> Res<T> op_prepare_argument(Vec<T>* v, bool padded) {
    // correlation.rs:96-117
    if (!v->is_complex || v->domain != 0) { mark_invalid(v); v->is_complex = 1; v->domain = 1; return done(v, 0); }
    if (padded) {
        const size_t points = points_of(v);
        if (points) {
            Res<T> r = op_zero_pad(v, 2 * points - 1, 1);
            if (r.result_code && points > 1) return r;
        }
    }
    Res<T> r = op_fft(v, false, false, false);
    if (r.result_code) return r;
    return op_complex_const(v, EW_CONJ, (T)0, (T)0);
}

template <typename T> Res<T> op_correlate(Vec<T>* v, const Vec<T>* other) {
    // correlation.rs:131-163
    if (v->domain != 0 || !v->is_complex || other->domain != 1 || !other->is_complex) {
        mark_invalid(v); v->is_complex = 1; v->domain = 1;
        return done(v, E_TIME);
    }
    const size_t points = points_of(other);
    const T delta = v->delta;
    Res<T> r = op_zero_pad(v, points, 1);
    if (r.result_code) return r;
    FftOpts f;
    int rc = ensure_scratch(v, v->len);
    if (!rc) rc = fft_exec<T>(v->d, v->scratch, points, 1, f, nullptr, 0, g_stream);
    if (rc) return done(v, rc);
    // mul(other), plain_ifft, scale(1/points), swap_halves (correlation.rs:151-160) as ONE transform: the product with the
    // prepared spectrum and the scale ride on the inverse transform's first load, swap_halves on its store
    FftOpts inv;
    inv.inverse = 1;
    inv.out_rot = points / 2;
    inv.in_mul.p = other->d; inv.in_mul.kind = 2;
    inv.scale = (double)((T)1 / (T)points);
    rc = fft_exec<T>(v->scratch, v->d, points, 1, inv, nullptr, 0, g_stream);
    v->delta = delta;
    return done(v, rc);
}

template <typename T> Res<T> op_reverse(Vec<T>* v) {
    const size_t n = points_of(v);
    if (n < 2) return done(v, 0);
    int rc = ensure_scratch(v, v->len);
    if (!rc) rc = ew_reverse<T>(v->d, v->scratch, n, v->is_complex ? 2 : 1, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    return done(v, 0);
}

template <typename T> Res<T> op_decimatei(Vec<T>* v, uint32_t factor, uint32_t delay) {
    const size_t n = points_of(v);
    if (factor == 0) return done(v, E_ARG_LEN);
    const size_t out = delay < n ? (n - delay + factor - 1) / factor : 0;
    const int esz = v->is_complex ? 2 : 1;
    if (out) {
        int rc = ensure_scratch(v, out * esz);
        if (!rc) rc = ew_decimate<T>(v->d, v->scratch, out, factor, delay, esz, g_stream);
        if (rc) return done(v, rc);
        trade(v);
    }
    v->len = out * esz;
    return done(v, 0);
}

// ---- interpolation ---------------------------------------------------------------------------------
// Shape and path of interpolatef (interpolation.rs:387-482) on `len` scalars, for the vector and the row API alike.
struct InterpfShape {
    size_t conv_len;     // clamped to half the points
    size_t new_len;      // output scalars: round(len * factor), made even
    size_t new_points;
    bool poly;           // polyphase tap tables with the integer factor F; else per-output taps
    int F;
};
template <typename T> int interpf_shape(size_t len, bool is_complex, T factor, size_t conv_len, InterpfShape* s) {
    const size_t points = is_complex ? len / 2 : len;
    s->conv_len = conv_len > points / 2 ? points / 2 : conv_len;
    const double nl = round((double)((T)len * factor));
    if (!(nl >= 0)) return E_ARG_LEN;
    s->new_len = (size_t)nl;
    s->new_len += s->new_len % 2;
    s->new_points = is_complex ? s->new_len / 2 : s->new_len;
    const bool integer = (T)fabs((T)round(factor) - factor) < (T)1e-6;
    s->poly = s->conv_len <= 202 && s->new_len >= 2000 && integer;
    s->F = s->poly ? (int)round(factor) : 0;
    return 0;
}

// Tap tables of the polyphase interpolatef path on the device: [2][F][2L+3] (interior, edge) over the window superset
// n = r-L-1+jj, jj in [0, 2L+3).
template <typename T> DeviceTable<T> interp_tap_tables(const RealFn<T>& f, T delay, int F, int L) {
    TableKey key = {};
    key.what = 2; key.a = (double)delay; key.n0 = (size_t)F; key.n1 = (size_t)L;
    return DeviceTable<T>(cache_key(f, &key), [&] {
        const int J = 2 * L + 3;
        // function_to_vectors (interpolation.rs:133-181): v_s[k] = f(j_k - s/F), j_0 = -(L-1) + delay
        std::vector<T> vs((size_t)F * (2 * L + 1));
        for (int s = 0; s < F; s++) {
            T offset = (T)s / (T)F;
            T j = -((T)L - (T)1) + delay;
            for (int k = 0; k < 2 * L + 1; k++) { vs[(size_t)s * (2 * L + 1) + k] = f(j - offset); j = j + (T)1; }
        }
        std::vector<T> tab((size_t)2 * F * J, (T)0);
        for (int s = 0; s < F; s++) {
            T* ti = &tab[(size_t)s * J];                    // interior (interpolation.rs:244-275)
            if (s == 0) { for (int jj = 0; jj <= 2 * L; jj++) ti[jj] = vs[2 * L - jj]; }
            else { for (int jj = 1; jj <= 2 * L + 1; jj++) ti[jj] = vs[(size_t)(F - s) * (2 * L + 1) + (2 * L + 1 - jj)]; }
            T* te = &tab[(size_t)(F + s) * J];              // edges (interpolation.rs:293-315)
            for (int k = 0; k <= 2 * L; k++) te[k + 2] = vs[(size_t)s * (2 * L + 1) + k];
        }
        return tab;
    });
}

template <typename T> Res<T> op_interpolatef(Vec<T>* v, const RealFn<T>& f, T factor, T delay, size_t conv_len) {
    // interpolation.rs:387-482
    delay = delay / v->delta;
    const size_t N = points_of(v);
    if (N == 0) return done(v, 0);
    InterpfShape s;
    int rc = interpf_shape<T>(v->len, v->is_complex != 0, factor, conv_len, &s);
    if (!rc) rc = ensure_scratch(v, s.new_len);
    if (rc) return done(v, rc);
    if (s.poly) {
        DeviceTable<T> tab = interp_tap_tables<T>(f, delay, s.F, (int)s.conv_len);
        rc = tab.rc ? tab.rc : interp_poly<T>(v->d, v->scratch, tab.p, N, s.new_points, s.F, (int)s.conv_len, v->is_complex, g_stream);
    } else {
        if (f.fn) return done(v, E_ARG_LEN);   // custom callback + per-output taps: not supported on the device
        rc = interp_frac<T>(v->d, v->scratch, N, s.new_points, (double)factor, (double)delay, (int)s.conv_len, f.kind,
                            (double)f.rolloff, v->is_complex, g_stream);
    }
    if (rc) return done(v, rc);
    trade(v);
    v->len = s.new_len;
    return done(v, 0);
}

template <typename T> std::vector<T> shifted_response_table(const RealFn<T>& f, bool is_symmetric, size_t points, T ratio) {
    std::vector<T> tab(points);
    const size_t offset = points % 2;
    const T mx = (T)(points - offset) / (T)2;
    const size_t c = (points - offset) / 2;
    auto val = [&](size_t i) {
        const T j = -mx + (T)i;
        const T xv = j <= (T)0 ? (T)1 + j / mx : -(mx - j + (T)1) / mx;
        return ratio * f(xv * ratio);
    };
    if (!is_symmetric) {
        for (size_t i = 0; i < points; i++) tab[i] = val(i);
    } else {
        for (size_t i = 0; i <= c; i++) tab[i] = val(i);
        if (offset == 0) { for (size_t i = 1; i < c; i++) tab[points - i] = tab[i]; }
        else { for (size_t i = 0; i < c; i++) tab[points - 1 - i] = tab[i]; }
    }
    return tab;
}

template <typename T> Res<T> op_interpolatei(Vec<T>* v, const RealFn<T>& f, bool is_symmetric, uint32_t factor) {
    // interpolation.rs:484-538: zero_interleave -> plain_fft -> * factor*f(shifted x * factor) -> plain_ifft ->
    // scale(1/points) (-> to_real).  The multiplier table follows multiply_function_priv with
    // is_fft_shifted = true, incl. the mirrored evaluation of symmetric functions.
    if (factor <= 1) return done(v, 0);
    if (!is_symmetric && !v->is_complex) return done(v, 10);   // ArgumentFunctionMustBeSymmetric
    const bool was_complex = v->is_complex != 0;
    const size_t n_in = points_of(v);
    if (!n_in) return done(v, 0);
    const size_t points = n_in * factor;
    // complex buffer of `points` points in the scratch: x[i] at i*factor, zeros elsewhere
    int rc = ensure_scratch(v, 2 * points);
    if (rc) return done(v, rc);
    if (was_complex) rc = ew_zero_interleave<T>(v->d, v->scratch, n_in, (int)factor, 2, g_stream);
    else rc = ew_zero_interleave<T>(v->d, v->scratch, n_in, (int)(2 * factor), 1, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    rc = ensure_scratch(v, 2 * points);
    if (rc) return done(v, rc);
    FftOpts fw;
    rc = fft_exec<T>(v->d, v->scratch, points, 1, fw, nullptr, 0, g_stream);
    if (rc) return done(v, rc);
    if (!f.fn) {
        // built-in responses (always symmetric): evaluated on the device (no O(points) host work, no table upload)
        rc = ew_mul_shifted_resp<T>(v->scratch, points, f.kind, (double)f.rolloff, (double)(T)factor, g_stream);
    } else {
        DeviceTable<T> tab(nullptr, [&] { return shifted_response_table<T>(f, is_symmetric, points, (T)factor); });
        rc = tab.rc ? tab.rc : ew_mul_table<T>(v->scratch, tab.p, points, 1, 0, g_stream);
    }
    if (rc) return done(v, rc);
    FftOpts inv;
    inv.inverse = 1;
    rc = fft_exec<T>(v->scratch, v->d, points, 1, inv, nullptr, 0, g_stream);
    if (!rc) rc = ew_scalar<T>(EW_SCALE, v->d, v->d, 2 * points, (double)((T)1 / (T)points), g_stream);
    if (rc) return done(v, rc);
    if (was_complex) { v->len = 2 * points; return done(v, 0); }
    rc = ew_complex_to_real<T>(C2R_REAL, v->d, v->scratch, points, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    v->len = points;
    return done(v, 0);
}


template <typename T> Res<T> op_interpolate(Vec<T>* v, const RealFn<T>* f, bool is_symmetric, size_t dest_points, T delay) {
    // interpolation.rs:541-604 (f == nullptr: interpft :533-539)
    if (f && !is_symmetric && !v->is_complex) return done(v, 10);   // ArgumentFunctionMustBeSymmetric
    const bool was_complex = v->is_complex != 0;
    const size_t n = points_of(v);
    if (!n || !dest_points) return done(v, E_ARG_LEN);
    const T delta_t = v->delta;
    const T factor = (T)dest_points / (T)n;
    int rc = 0;
    if (!was_complex) {
        rc = ensure_scratch(v, 2 * n);
        if (!rc) rc = ew_zero_interleave<T>(v->d, v->scratch, n, 2, 1, g_stream);
        if (rc) return done(v, rc);
        trade(v);
    }
    const size_t big = 2 * (n > dest_points ? n : dest_points);
    rc = ensure_scratch(v, big);
    FftOpts fw;
    if (!rc) rc = fft_exec<T>(v->d, v->scratch, n, 1, fw, nullptr, 0, g_stream);
    if (!rc) rc = reserve(&v->d, &v->cap, big, false, 0);
    if (rc) return done(v, rc);
    // spectrum in the scratch -> re-binned spectrum in d
    std::optional<DeviceTable<T>> tab;
    double scale = 1.0;
    int use_scale = 0;
    int resp_kind = -1;
    if (dest_points > n) {
        if (f && !f->fn) resp_kind = f->kind;      // built-in response (always symmetric): evaluated on the device
        else if (f) {
            tab.emplace(nullptr, [&] { return shifted_response_table<T>(*f, is_symmetric, dest_points, factor); });
            if (tab->rc) return done(v, tab->rc);
        } else { scale = (double)factor; use_scale = 1; }
    } else if (dest_points < n) {
        scale = (double)((T)(2 * dest_points) / (T)(2 * n));
        use_scale = 1;
    }
    const T pi = (T)M_PI;
    const T phase_inc = (T)2 * pi * (delay / delta_t) / (T)n;
    rc = ew_resample_spectrum<T>(v->scratch, v->d, n, dest_points, tab ? tab->p : nullptr, scale, use_scale, (double)phase_inc, delay != (T)0, resp_kind,
                                 f ? (double)f->rolloff : 0.0, (double)factor, g_stream);
    if (rc) return done(v, rc);
    FftOpts inv;
    inv.inverse = 1;
    inv.scale = (double)((T)1 / (T)dest_points);
    rc = fft_exec<T>(v->d, v->scratch, dest_points, 1, inv, nullptr, 0, g_stream);
    if (rc) return done(v, rc);
    if (was_complex) {
        trade(v);
        v->len = 2 * dest_points;
    } else {
        rc = ew_complex_to_real<T>(C2R_REAL, v->scratch, v->d, dest_points, g_stream);
        if (rc) return done(v, rc);
        v->len = dest_points;
    }
    v->delta = delta_t / factor;
    return done(v, 0);
}

template <typename T> Res<T> op_mul_cexp(Vec<T>* v, T a, T b) {
    if (!v->is_complex) { mark_invalid(v); return done(v, 0); }
    const T aa = a * v->delta, bb = b * v->delta;
    return done(v, ew_mul_cexp<T>(v->d, points_of(v), (double)aa, (double)bb, g_stream));
}

template <typename T> Res<T> op_mirror(Vec<T>* v) {
    // freq.rs:52-83
    if (v->domain != 1 && !v->is_complex) { mark_invalid(v); return done(v, 0); }
    const size_t p = v->len / 2;
    if (!p) return done(v, 0);
    int rc = ensure_scratch(v, 2 * (2 * p - 1));
    if (!rc) rc = ew_mirror<T>(v->d, v->scratch, p, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    v->len = 2 * (2 * p - 1);
    return done(v, 0);
}

template <typename T> Res<T> op_sfft(Vec<T>* v, bool shifted, const WinFn<T>* window) {
    // time_to_freq.rs:197-298; kept length follows the statically typed vectors: (n + 1) / 2 complex points
    if (v->domain != 0 || v->is_complex) {
        mark_invalid(v); v->is_complex = 1; v->domain = 1;
        return done(v, E_TIME);
    }
    const size_t n = v->len;
    if (n % 2 == 0) {
        mark_invalid(v); v->is_complex = 1; v->domain = 1;
        return done(v, 9);   // InputMustHaveAnOddLength
    }
    if (window) {
        Res<T> r = op_window_fn(v, *window, false);
        if (r.result_code) return r;
    }
    Res<T> r = op_fft(v, false, shifted, false);
    if (r.result_code) return r;
    v->len = n + 1;
    // The DC bin of a real signal is real.  Mixed-radix transforms deliver an exact zero there (which
    // plain_sifft's |Im X[0]| <= 1e-10 test relies on, freq_to_time.rs:204); the chirp-z path used for
    // general odd lengths leaves rounding noise, so the exact value is stored.
    const size_t dc = shifted ? (n - 1) / 2 : 0;
    cudaError_t e = cudaMemsetAsync(v->d + 2 * dc + 1, 0, sizeof(T), g_stream);
    if (e != cudaSuccess) { set_last_error("sfft: %s", cudaGetErrorString(e)); return done(v, -1000 - (int)e); }
    return done(v, 0);
}

template <typename T> Res<T> op_sifft(Vec<T>* v, bool shifted, const WinFn<T>* window) {
    // freq_to_time.rs:190-248
    if (shifted) {
        const size_t points = points_of(v);
        if (points) {
            int rc = ew_scalar<T>(EW_SCALE, v->d, v->d, v->len, (double)((T)1 / (T)points), g_stream);
            if (rc) return done(v, rc);
        }
        Res<T> r = op_rotate(v, false);
        if (r.result_code) return r;
    }
    if (v->domain != 1 || !v->is_complex) {
        mark_invalid(v); v->is_complex = 1; v->domain = 1;
        return done(v, E_FREQ);
    }
    const size_t p = points_of(v);
    if (p) {
        T im0 = 0;
        cudaError_t e = cudaMemcpyAsync(&im0, v->d + 1, sizeof(T), cudaMemcpyDeviceToHost, g_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_stream);
        if (e != cudaSuccess) { set_last_error("plain_sifft: %s", cudaGetErrorString(e)); return done(v, -1000 - (int)e); }
        if (fabs((double)im0) > 1e-10) {
            mark_invalid(v); v->is_complex = 1; v->domain = 1;
            return done(v, 8);   // InputMustBeConjSymmetric
        }
    }
    Res<T> r = op_mirror(v);
    if (r.result_code) return r;
    r = op_fft(v, true, false, false);
    if (r.result_code) return r;
    const size_t points = points_of(v);
    if (points) {
        int rc = ensure_scratch(v, points);
        if (!rc) rc = ew_complex_to_real<T>(C2R_REAL, v->d, v->scratch, points, g_stream);
        if (rc) return done(v, rc);
        trade(v);
    }
    v->len = points;
    v->is_complex = 0;
    v->domain = 0;
    if (window) return op_window_fn(v, *window, true);
    return done(v, 0);
}

template <typename T> Res<T> op_interpolate_lin(Vec<T>* v, T factor, T delay) {
    // real_interpolation.rs:33-71
    if (v->is_complex) { mark_invalid(v); return done(v, 0); }
    const size_t n = v->len;
    if (n == 0) return done(v, 0);
    const size_t dest_len = (size_t)round((double)((T)(n - 1) * factor)) + 1;
    int rc = ensure_scratch(v, dest_len);
    if (!rc) rc = interp_lin<T>(v->d, v->scratch, n, dest_len, (double)factor, (double)delay, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    v->len = dest_len;
    return done(v, 0);
}


// ---- SURVEY 8(f) row 4: the rest of the C facade (elementwise math, reorganisation, reductions) -------
template <typename T> Res<T> op_math(Vec<T>* v, int op, T arg, bool real_only) {
    // trigonometry_and_powers.rs:198-377; real_only: assert_real! (real_ops.rs:227-234)
    if (real_only && v->is_complex) { mark_invalid(v); return done(v, 0); }
    return done(v, math_unary<T>(op, v->d, points_of(v), v->is_complex, (double)arg, g_stream));
}

template <typename T> Res<T> op_unwrap(Vec<T>* v, T divisor) {
    if (v->is_complex) { mark_invalid(v); return done(v, 0); }
    return done(v, math_unwrap<T>(v->d, v->len, (double)divisor, g_stream));
}

template <typename T> Res<T> op_diff(Vec<T>* v, bool with_start) {
    // diff_sum.rs:63-109
    const size_t step = v->is_complex ? 2 : 1;
    if (v->len < step) return done(v, 0);
    const size_t n_out = with_start ? v->len : v->len - step;
    int rc = ensure_scratch(v, v->len);
    if (!rc) rc = math_diff<T>(v->d, v->scratch, n_out, (int)step, with_start, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    v->len = n_out;
    return done(v, 0);
}

template <typename T> Res<T> op_cum_sum(Vec<T>* v) {
    // diff_sum.rs:111-122 (the running sum is evaluated as a parallel scan: same value up to rounding order)
    const int lanes = v->is_complex ? 2 : 1;
    const size_t points = points_of(v);
    if (!points) return done(v, 0);
    int rc = ensure_scratch(v, v->len);
    if (rc) return done(v, rc);
    void* work = workspace(math_cumsum_workspace(points, lanes, sizeof(T)), 3);
    if (!work) return done(v, -1001);
    rc = math_cumsum<T>(v->d, v->scratch, work, points, lanes, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    return done(v, 0);
}

template <typename T> Res<T> op_binary_smaller(Vec<T>* v, const Vec<T>* o, int op) {
    // elementary.rs:457-517,601-639
    if (o->len == 0 || v->len % o->len != 0) return done(v, E_ARG_LEN);
    if (!meta_agrees(v, o)) return done(v, E_META);
    return done(v, math_binary_smaller<T>(op, v->d, o->d, points_of(v), points_of(o), v->is_complex, g_stream));
}

template <typename T> Res<T> op_set_pair(Vec<T>* v, const Vec<T>* a, const Vec<T>* b, bool polar) {
    // complex_to_real.rs:726-770
    if (a->len != b->len) return done(v, E_ARG_LEN);
    const size_t points = a->len;
    int rc = reserve(&v->d, &v->cap, 2 * points, false, 0);
    if (!rc) rc = math_compose<T>(a->d, b->d, v->d, points, polar, g_stream);
    if (rc) return done(v, rc);
    v->len = 2 * points;
    return done(v, 0);
}

template <typename T> int32_t op_get_real_imag(Vec<T>* v, Vec<T>* re, Vec<T>* im) {
    // complex_to_real.rs:674-691
    if (!v->is_complex || re->is_complex || im->is_complex) {
        re->len = 0; im->len = 0; re->version++; im->version++;
        return VOID_OK;
    }
    const size_t points = v->len / 2;
    vec_resize(re, points);
    vec_resize(im, points);
    if (points) {
        int rc = ew_complex_to_real<T>(C2R_REAL, v->d, re->d, points, g_stream);
        if (!rc) rc = ew_complex_to_real<T>(C2R_IMAG, v->d, im->d, points, g_stream);
        if (rc) return rc;
    }
    return VOID_OK;
}

template <typename T> int32_t op_split_into(const Vec<T>* v, Vec<T>** targets, size_t n) {
    // data_reorganization.rs:484-512
    if (n == 0 || v->len % n != 0) return E_ARG_LEN;
    const size_t part_len = v->len / n;
    std::vector<void*> ptrs(n);
    for (size_t i = 0; i < n; i++) {
        int rc = vec_resize(targets[i], part_len);
        if (rc) return rc;
        ptrs[i] = targets[i]->d;
    }
    const int esz = v->is_complex ? 2 : 1;
    int rc = math_split_merge<T>(v->d, ptrs.data(), (int)n, v->len / esz, esz, 0, g_stream);
    return rc ? rc : VOID_OK;
}

template <typename T> Res<T> op_merge(Vec<T>* v, Vec<T>* const* sources, size_t n) {
    // data_reorganization.rs:522-557
    if (n == 0) return done(v, E_ARG_LEN);
    for (size_t i = 1; i < n; i++) if (sources[i]->len != sources[0]->len) return done(v, E_ARG_LEN);
    int rc = vec_resize(v, sources[0]->len * n);
    if (rc) return done(v, rc);
    std::vector<void*> ptrs(n);
    for (size_t i = 0; i < n; i++) ptrs[i] = sources[i]->d;
    const int esz = v->is_complex ? 2 : 1;
    return done(v, math_split_merge<T>(v->d, ptrs.data(), (int)n, v->len / esz, esz, 1, g_stream));
}

template <typename T> Res<T> op_interpolate_hermite(Vec<T>* v, T factor, T delay) {
    // real_interpolation.rs:73-178
    if (v->is_complex) { mark_invalid(v); return done(v, 0); }
    const size_t n = v->len;
    if (n < 3) return done(v, E_ARG_LEN);
    const size_t dest_len = (size_t)round((double)((T)(n - 1) * factor)) + 1;
    const double st = ceil((double)(((T)1 - delay) * factor));
    const size_t start = st < 0 ? 0 : (size_t)st;
    int rc = ensure_scratch(v, dest_len);
    if (!rc) rc = math_hermite<T>(v->d, v->scratch, n, dest_len, start, (double)factor, (double)delay, g_stream);
    if (rc) return done(v, rc);
    trade(v);
    v->len = dest_len;
    return done(v, 0);
}

// reductions: values in double, converted by the facade to the reference's result types
template <typename T> int sums_of(const Vec<T>* v, int prec, double* out4) {
    out4[0] = out4[1] = out4[2] = out4[3] = 0.0;
    if (!v->len) return 0;
    return reduce_sums<T>(v->d, points_of(v), v->is_complex, prec, out4, g_stream);
}

template <typename T> int dot_of(const Vec<T>* v, const Vec<T>* o, bool want_complex, int prec, double* out2) {
    // dot_products.rs:67-160, 289-345
    out2[0] = out2[1] = 0.0;
    if (want_complex) {
        if (!v->is_complex) return E_COMPLEX;
        if (!o->is_complex || v->domain != o->domain) return E_META;
    } else if (v->is_complex) return E_REAL;
    const size_t n = v->len < o->len ? v->len : o->len;
    const size_t elems = want_complex ? n / 2 : n;
    if (!elems) return 0;
    return reduce_dot<T>(v->d, o->d, elems, want_complex, prec, out2, g_stream);
}

template <typename S> void stats_fill_real(S* out, const StatsRaw& r) {
    typedef decltype(out->sum) V;
    const double n = (double)r.count;
    out->sum = (V)r.sum[0]; out->count = (size_t)r.count;
    out->average = (V)((V)r.sum[0] / (V)n);
    out->rms = (V)sqrt((double)((V)r.sumsq[0] / (V)n));
    out->min = (V)r.min[0]; out->min_index = (size_t)r.min_index;
    out->max = (V)r.max[0]; out->max_index = (size_t)r.max_index;
}
template <typename S, typename V> void stats_fill_complex(S* out, const StatsRaw& r) {
    const V n = (V)r.count;
    out->sum.re = (V)r.sum[0]; out->sum.im = (V)r.sum[1]; out->count = (size_t)r.count;
    out->average.re = (V)r.sum[0] / n; out->average.im = (V)r.sum[1] / n;
    // rms = sqrt(sum(z^2) / count), complex square root as in num-complex (principal branch)
    const double qr = (double)((V)r.sumsq[0] / n), qi = (double)((V)r.sumsq[1] / n);
    double sr, si;
    if (qi == 0.0) { if (qr >= 0) { sr = sqrt(qr); si = qi; } else { sr = 0; si = sqrt(-qr); } }
    else if (qr == 0.0) { const double x = sqrt(fabs(qi) / 2); sr = x; si = qi < 0 ? -x : x; }
    else { const double m = sqrt(hypot(qr, qi)), th = atan2(qi, qr) / 2; sr = m * cos(th); si = m * sin(th); }
    out->rms.re = (V)sr; out->rms.im = (V)si;
    out->min.re = (V)r.min[0]; out->min.im = (V)r.min[1]; out->min_index = (size_t)r.min_index;
    out->max.re = (V)r.max[0]; out->max.im = (V)r.max[1]; out->max_index = (size_t)r.max_index;
}

template <typename T> int stats_of(const Vec<T>* v, int parts, int prec, StatsRaw* raw) {
    // statistics.rs:179-440; an empty vector yields the reference's empty record (count 0, NaN average / rms)
    for (int p = 0; p < parts; p++) {
        raw[p] = StatsRaw();
        raw[p].min[0] = INFINITY; raw[p].min[1] = v->is_complex ? INFINITY : 0.0;
        raw[p].max[0] = v->is_complex ? 0.0 : -INFINITY;
    }
    if (!v->len) return 0;
    return reduce_stats<T>(v->d, points_of(v), v->is_complex, parts, prec, raw, g_stream);
}

// ---- host access -----------------------------------------------------------------------------------
template <typename T> const T* host_mirror(const Vec<T>* cv) {
    Vec<T>* v = const_cast<Vec<T>*>(cv);
    v->host.resize(v->len ? v->len : 1);
    if (v->len) {
        cudaMemcpyAsync(v->host.data(), v->d, v->len * sizeof(T), cudaMemcpyDeviceToHost, g_stream);
        cudaStreamSynchronize(g_stream);
    }
    return v->host.data();
}

template <typename T> int upload(Vec<T>* v, const T* host, size_t len) {
    if (len != v->len) {
        int rc = vec_resize(v, len);
        if (rc) return rc;
    }
    if (len) BDSP_CUDA_OK(cudaMemcpyAsync(v->d, host, len * sizeof(T), cudaMemcpyHostToDevice, g_stream));
    v->version++;
    return 0;
}
template <typename T> int download(const Vec<T>* v, T* host, size_t len, bool wait) {
    if (len > v->len) return E_ARG_LEN;
    if (len) BDSP_CUDA_OK(cudaMemcpyAsync(host, v->d, len * sizeof(T), cudaMemcpyDeviceToHost, g_stream));
    if (wait) BDSP_CUDA_OK(cudaStreamSynchronize(g_stream));
    return 0;
}


// ---- host callbacks per element (mapping.rs:46-266; facade32.rs:594-647) -----------------------------
// The computation IS the caller's host function, so the vector is staged through its host mirror: download,
// apply the callback in index order, upload.  (No device work besides the two copies.)
template <typename T> Res<T> op_map_inplace_real(Vec<T>* v, T (*map)(T, size_t)) {
    if (v->is_complex) { mark_invalid(v); return done(v, 0); }
    host_mirror(v);
    for (size_t i = 0; i < v->len; i++) v->host[i] = map(v->host[i], i);
    int rc = upload(v, v->host.data(), v->len);
    if (!rc) { cudaError_t e = cudaStreamSynchronize(g_stream); if (e != cudaSuccess) rc = -1000 - (int)e; }
    return done(v, rc);
}
template <typename T, typename CT> Res<T> op_map_inplace_complex(Vec<T>* v, CT (*map)(CT, size_t)) {
    if (!v->is_complex) { mark_invalid(v); return done(v, 0); }
    host_mirror(v);
    CT* c = reinterpret_cast<CT*>(v->host.data());
    for (size_t i = 0; i < v->len / 2; i++) c[i] = map(c[i], i);
    int rc = upload(v, v->host.data(), v->len);
    if (!rc) { cudaError_t e = cudaStreamSynchronize(g_stream); if (e != cudaSuccess) rc = -1000 - (int)e; }
    return done(v, rc);
}
template <typename T, typename ET> BdspPointerResult op_map_aggregate(const Vec<T>* v, bool complex_variant, const void* (*map)(ET, size_t),
                                                                      const void* (*aggregate)(const void*, const void*)) {
    BdspPointerResult out; out.result_code = 0; out.result = nullptr;
    if (complex_variant != (v->is_complex != 0)) { out.result_code = complex_variant ? E_COMPLEX : E_REAL; return out; }
    if (v->len == 0) { out.result_code = 12; return out; }   // InputMustNotBeEmpty
    const ET* h = reinterpret_cast<const ET*>(host_mirror(v));
    const size_t n = complex_variant ? v->len / 2 : v->len;
    const void* acc = map(h[0], 0);
    for (size_t i = 1; i < n; i++) acc = aggregate(acc, map(h[i], i));
    out.result = acc;
    if (erroneous(v)) out.result_code = -1;
    return out;
}

template <typename T>
int scale_mul_mag_phase(Vec<T>* v, T cre, T cim, const Vec<T>* w, Vec<T>* mag, Vec<T>* ph, int write_back) {
    if (!v->is_complex || !w->is_complex) return E_COMPLEX;
    if (mag->is_complex || ph->is_complex) return E_REAL;
    if (v->len != w->len) return E_SAME_SIZE;
    if (!meta_agrees(v, w)) return E_META;
    const size_t points = v->len / 2;
    int rc = vec_resize(mag, points);
    if (!rc) rc = vec_resize(ph, points);
    if (rc) return rc;
    mag->delta = v->delta; ph->delta = v->delta;
    if (points) rc = ew_scale_mul_mag_phase<T>(v->d, w->d, mag->d, ph->d, points, (double)cre, (double)cim, cim != (T)0, write_back, g_stream);
    if (write_back) v->version++;
    return rc;
}

struct ConvPlan {
    int is64;
    size_t L;
    OlsPlan* ols;   // overlap-save plan of the taps, where convolve() needs one
    void* taps;     // copy of the taps (L complex)
};

template <typename T> ConvPlan* conv_plan_create(const void* h_dev, size_t L) {
    typedef typename CpxOf<T>::type C;
    if (!h_dev || !L) { set_last_error("conv plan: empty impulse response"); return nullptr; }
    ConvPlan* p = new ConvPlan();
    p->is64 = sizeof(T) == 8; p->L = L; p->ols = nullptr; p->taps = nullptr;
    if (cudaMalloc(&p->taps, L * sizeof(C)) != cudaSuccess) { delete p; return nullptr; }
    cudaMemcpyAsync(p->taps, h_dev, L * sizeof(C), cudaMemcpyDeviceToDevice, g_stream);
    if (conv_needs_plan<T>(L, 0)) {
        p->ols = ols_plan_create<T>(p->taps, L, 0, true, g_stream);
        if (!p->ols) { cudaFree(p->taps); delete p; return nullptr; }
    }
    return p;
}

template <typename T> int conv_rows(const void* in, void* out, size_t points, size_t rows, const ConvPlan* p) {
    if (!p || p->is64 != (sizeof(T) == 8)) { set_last_error("conv rows: plan precision mismatch"); return -2; }
    if (points < p->L) return E_ARG_LEN;
    if (!points || !rows) return 0;
    return convolve<T>(in, out, points, rows, 0, p->taps, p->L, 0, p->ols, g_stream);
}

template <typename T> int fft_rows(const void* in, void* out, size_t points, size_t rows, int flags) {
    const bool inverse = (flags & BDSP_F_INVERSE) != 0;
    const int wk = (flags >> 8) & 15;   // BDSP_F_WINDOW(kind): every row is multiplied by the window on the way in (windowed_fft per row)
    if (wk && inverse) { set_last_error("fft rows: a window applies to forward transforms only"); return -2; }
    const FftOpts o = fft_opts<T>(points, inverse, (flags & BDSP_F_SHIFT) != 0, (flags & BDSP_F_MAGNITUDE) != 0,
                                  (flags & BDSP_F_REAL_INPUT) != 0, wk ? wk - 1 : RECTANGULAR);
    return fft_exec<T>(in, out, points, rows, o, nullptr, 0, g_stream);
}

// fft_rows over `frames` frames of one signal, frame f = the `points` points from point f*hop on (short-time analysis)
template <typename T> int fft_frames(const void* in, void* out, size_t points, size_t hop, size_t frames, int flags) {
    if (flags & BDSP_F_INVERSE) { set_last_error("fft frames: frames are analysis frames, BDSP_F_INVERSE is not accepted"); return -2; }
    if (!hop) { set_last_error("fft frames: hop must be at least 1"); return -2; }
    if (!points || !frames) return 0;
    const bool real = (flags & BDSP_F_REAL_INPUT) != 0, mag = (flags & BDSP_F_MAGNITUDE) != 0;
    const size_t in_esz = real ? sizeof(T) : 2 * sizeof(T), out_esz = mag ? sizeof(T) : 2 * sizeof(T);
    const size_t max = ~(size_t)0;
    if (frames - 1 > (max - points) / hop || ((frames - 1) * hop + points) > max / in_esz || frames > max / points / out_esz) {
        set_last_error("fft frames: %zu frames of %zu points, hop %zu overflow the address space", frames, points, hop);
        return -2;
    }
    const uintptr_t i0 = reinterpret_cast<uintptr_t>(in), o0 = reinterpret_cast<uintptr_t>(out);
    const size_t in_bytes = ((frames - 1) * hop + points) * in_esz, out_bytes = frames * points * out_esz;
    if (i0 < o0 + out_bytes && o0 < i0 + in_bytes) { set_last_error("fft frames: the output overlaps the input"); return -3; }
    const int wk = (flags >> 8) & 15;
    FftOpts o = fft_opts<T>(points, false, (flags & BDSP_F_SHIFT) != 0, mag, real, wk ? wk - 1 : RECTANGULAR);
    o.in_stride = hop;
    return fft_exec<T>(in, out, points, frames, o, nullptr, 0, g_stream);
}

// the inverse of fft_frames: inverse rows scaled by 1/points, then the least-squares overlap-add of the frames under the
// synthesis window (torch.istft(center=False), scipy.signal.istft) into (frames-1)*hop + points points
template <typename T> int ifft_frames(const void* in, void* out, size_t points, size_t hop, size_t frames, int flags) {
    const int unknown = flags & ~(BDSP_F_SHIFT | BDSP_F_REAL_OUTPUT | (15 << 8));   // (15 << 8): every BDSP_F_WINDOW(kind)
    if (unknown) {
        const char* name = (unknown & BDSP_F_INVERSE) ? "BDSP_F_INVERSE" : (unknown & BDSP_F_MAGNITUDE) ? "BDSP_F_MAGNITUDE"
                         : (unknown & BDSP_F_REAL_INPUT) ? "BDSP_F_REAL_INPUT" : nullptr;
        if (name) set_last_error("ifft frames: %s is not accepted (BDSP_F_SHIFT, BDSP_F_REAL_OUTPUT, BDSP_F_WINDOW(kind) are)", name);
        else set_last_error("ifft frames: unknown flag bits 0x%x", (unsigned)unknown);
        return -2;
    }
    if (!hop) { set_last_error("ifft frames: hop must be at least 1"); return -2; }
    if (!points || !frames) return 0;
    if (hop > points) { set_last_error("ifft frames: hop %zu > %zu points leaves samples that no frame covers", hop, points); return -2; }
    const bool real_out = (flags & BDSP_F_REAL_OUTPUT) != 0;
    const size_t in_esz = 2 * sizeof(T), out_esz = real_out ? sizeof(T) : 2 * sizeof(T);
    // hop <= points: the output's (frames-1)*hop + points points are at most the input's frames*points
    if (frames > ~(size_t)0 / points / in_esz) {
        set_last_error("ifft frames: %zu frames of %zu points overflow the address space", frames, points);
        return -2;
    }
    const uintptr_t i0 = reinterpret_cast<uintptr_t>(in), o0 = reinterpret_cast<uintptr_t>(out);
    const size_t in_bytes = frames * points * in_esz, out_bytes = ((frames - 1) * hop + points) * out_esz;
    if (i0 < o0 + out_bytes && o0 < i0 + in_bytes) { set_last_error("ifft frames: the output overlaps the input"); return -3; }
    const int wk = (flags >> 8) & 15;
    FftOpts o = fft_opts<T>(points, true, (flags & BDSP_F_SHIFT) != 0, false, false, wk ? wk - 1 : RECTANGULAR);
    o.scale = (double)((T)1 / (T)points);   // ifft()'s 1/points, with or without the shift
    return ifft_frames_exec<T>(in, out, points, hop, frames, o, real_out, g_stream);
}

// The checks shared by the averaged-spectrum entry points (welch, csd, coherence), in this order: the flags (`known` are
// accepted and listed in `accepted`; any other is named), BDSP_F_ONESIDED only with BDSP_F_REAL_INPUT and without
// BDSP_F_SHIFT, hop >= 1, fs finite and > 0 where it is used, sizes that fit size_t.  Returns -2 with bdsp_last_error set,
// or 0 with the byte counts of one input signal and of the output (out_esz bytes per output value); both 0 for an empty
// call (points or frames 0).
template <typename T>
int spectrum_args(const char* fn, int flags, int known, const char* accepted, size_t points, size_t hop, size_t frames, bool fs_used,
                  double fs, size_t out_esz, size_t* in_bytes, size_t* out_bytes) {
    *in_bytes = *out_bytes = 0;
    const int unknown = flags & ~known;
    if (unknown) {
        const char* name = (unknown & BDSP_F_INVERSE) ? "BDSP_F_INVERSE" : (unknown & BDSP_F_MAGNITUDE) ? "BDSP_F_MAGNITUDE"
                         : (unknown & BDSP_F_REAL_OUTPUT) ? "BDSP_F_REAL_OUTPUT" : (unknown & BDSP_F_POWER_SPECTRUM) ? "BDSP_F_POWER_SPECTRUM"
                         : nullptr;
        if (name) set_last_error("%s: %s is not accepted (%s are)", fn, name, accepted);
        else set_last_error("%s: unknown flag bits 0x%x", fn, (unsigned)unknown);
        return -2;
    }
    const bool real = (flags & BDSP_F_REAL_INPUT) != 0, shift = (flags & BDSP_F_SHIFT) != 0, onesided = (flags & BDSP_F_ONESIDED) != 0;
    if (onesided && !real) { set_last_error("%s: BDSP_F_ONESIDED needs BDSP_F_REAL_INPUT (a complex signal has no symmetric spectrum)", fn); return -2; }
    if (onesided && shift) { set_last_error("%s: BDSP_F_ONESIDED and BDSP_F_SHIFT exclude each other", fn); return -2; }
    if (!hop) { set_last_error("%s: hop must be at least 1", fn); return -2; }
    if (fs_used && !(isfinite(fs) && fs > 0)) { set_last_error("%s: the sampling rate fs must be finite and > 0", fn); return -2; }
    if (!points || !frames) return 0;
    const size_t in_esz = real ? sizeof(T) : 2 * sizeof(T);
    const size_t max = ~(size_t)0;
    if (frames - 1 > (max - points) / hop || ((frames - 1) * hop + points) > max / in_esz || points > max / out_esz) {
        set_last_error("%s: %zu frames of %zu points, hop %zu overflow the address space", fn, frames, points, hop);
        return -2;
    }
    *in_bytes = ((frames - 1) * hop + points) * in_esz;
    *out_bytes = (onesided ? points / 2 + 1 : points) * out_esz;
    return 0;
}

static bool ranges_overlap(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(a), b0 = reinterpret_cast<uintptr_t>(b);
    return a0 < b0 + b_bytes && b0 < a0 + a_bytes;
}

// Welch's averaged periodogram of a signal's frames (scipy.signal.welch with detrend=False, MATLAB pwelch): the frames of
// fft_frames, |X|^2 averaged over them and scaled as a density or a power spectrum, two-sided or one-sided
template <typename T> int welch(const void* in, void* out, size_t points, size_t hop, size_t frames, int flags, double fs) {
    const int known = BDSP_F_REAL_INPUT | BDSP_F_SHIFT | (15 << 8) | BDSP_F_ONESIDED | BDSP_F_POWER_SPECTRUM;   // (15 << 8): BDSP_F_WINDOW(kind)
    const bool power = (flags & BDSP_F_POWER_SPECTRUM) != 0;
    size_t in_bytes, out_bytes;
    const int rc = spectrum_args<T>("welch", flags, known, "BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED, BDSP_F_POWER_SPECTRUM",
                                    points, hop, frames, !power, fs, sizeof(T), &in_bytes, &out_bytes);
    if (rc || !in_bytes) return rc;
    if (ranges_overlap(in, in_bytes, out, out_bytes)) { set_last_error("welch: the output overlaps the input"); return -3; }
    const int wk = (flags >> 8) & 15;
    const FftOpts o = fft_opts<T>(points, false, (flags & BDSP_F_SHIFT) != 0, false, (flags & BDSP_F_REAL_INPUT) != 0, wk ? wk - 1 : RECTANGULAR);
    return welch_exec<T>(in, static_cast<T*>(out), points, hop, frames, o, (flags & BDSP_F_ONESIDED) != 0, power, fs, g_stream);
}

// Cross-spectral density (scipy.signal.csd with detrend=False) or, with `coherence`, the magnitude-squared coherence
// (scipy.signal.coherence) of two signals' frames, each framed as welch frames its input.  x and y are only read, so they
// may be the same buffer; the output may overlap neither.
template <typename T> int cross_spectrum(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int flags,
                                         double fs, bool coherence) {
    const char* fn = coherence ? "coherence" : "csd";
    const int known = BDSP_F_REAL_INPUT | BDSP_F_SHIFT | (15 << 8) | BDSP_F_ONESIDED | (coherence ? 0 : BDSP_F_POWER_SPECTRUM);
    const bool power = (flags & BDSP_F_POWER_SPECTRUM) != 0;
    size_t in_bytes, out_bytes;
    const int rc = spectrum_args<T>(fn, flags, known, coherence ? "BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED"
                                                                : "BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED, BDSP_F_POWER_SPECTRUM",
                                    points, hop, frames, !coherence && !power, fs, coherence ? sizeof(T) : 2 * sizeof(T), &in_bytes, &out_bytes);
    if (rc || !in_bytes) return rc;
    if (ranges_overlap(x, in_bytes, out, out_bytes)) { set_last_error("%s: the output overlaps x", fn); return -3; }
    if (ranges_overlap(y, in_bytes, out, out_bytes)) { set_last_error("%s: the output overlaps y", fn); return -3; }
    const int wk = (flags >> 8) & 15;
    const FftOpts o = fft_opts<T>(points, false, (flags & BDSP_F_SHIFT) != 0, false, (flags & BDSP_F_REAL_INPUT) != 0, wk ? wk - 1 : RECTANGULAR);
    return csd_exec<T>(x, y, out, points, hop, frames, o, (flags & BDSP_F_ONESIDED) != 0, power, fs, coherence, g_stream);
}

// ---- batched (matrix-row) forms: the reference's MatrixMxN applies the vector operation to every row in turn
// (matrix/src/time_freq.rs:52-74, matrix/src/complex.rs:18-26); rows sit back to back in device memory ----------------------
// magnitude (hypot, complex_to_real.rs:376) / phase (atan2, :402) / magnitude_squared of `rows` rows: elementwise, so the
// batch is one launch over rows * points points
template <typename T> int c2r_rows(int op, const void* in, void* out, size_t points, size_t rows) {
    if (!points || !rows) return 0;
    return ew_complex_to_real<T>(op, in, out, points * rows, g_stream);
}
// fused scale(c) -> mul(&w) -> (magnitude, phase) over rows (elementwise as well; w has the same shape as v)
template <typename T>
int chain_rows(void* v, const void* w, void* mag, void* phase, size_t points, size_t rows, T cre, T cim, int write_back) {
    if (!points || !rows) return 0;
    return ew_scale_mul_mag_phase<T>(v, w, mag, phase, points * rows, (double)cre, (double)cim, cim != (T)0, write_back, g_stream);
}
// interpolatef (interpolation.rs:387-482) with a built-in impulse response on `rows` rows of `points` points (complex or
// real): the polyphase path's tap tables are built once, every row is one kernel launch.
// out: rows * new_points points, new_points as interpolatef32 computes it.  Returns the reference's error codes.
template <typename T>
int interp_rows(const void* in, void* out, size_t points, size_t rows, int is_complex, int kind, T rolloff, T factor, T delay,
                size_t conv_len, size_t* new_points_out) {
    typedef typename CpxOf<T>::type C;
    InterpfShape s;
    int rc = interpf_shape<T>(is_complex ? 2 * points : points, is_complex != 0, factor, conv_len, &s);
    if (rc) return rc;
    if (new_points_out) *new_points_out = s.new_points;
    if (!points || !rows) return 0;
    RealFn<T> f;
    f.kind = kind == 0 ? 0 : 1;
    f.rolloff = rolloff;
    const size_t esz = is_complex ? sizeof(C) : sizeof(T);
    const char* x = reinterpret_cast<const char*>(in);
    char* y = reinterpret_cast<char*>(out);
    const int L = (int)s.conv_len;
    if (s.poly) {
        DeviceTable<T> tab = interp_tap_tables<T>(f, delay, s.F, L);
        rc = tab.rc;
        for (size_t r = 0; r < rows && !rc; r++)
            rc = interp_poly<T>(x + r * esz * points, y + r * esz * s.new_points, tab.p, points, s.new_points, s.F, L, is_complex, g_stream);
        return rc;
    }
    for (size_t r = 0; r < rows && !rc; r++)
        rc = interp_frac<T>(x + r * esz * points, y + r * esz * s.new_points, points, s.new_points, (double)factor, (double)delay, L,
                            f.kind, (double)rolloff, is_complex, g_stream);
    return rc;
}

}  // namespace

// =====================================================================================================
// extern "C" surface
// =====================================================================================================
#define V32(p) reinterpret_cast<Vec<float>*>(p)
#define V64(p) reinterpret_cast<Vec<double>*>(p)
#define CV32(p) reinterpret_cast<const Vec<float>*>(p)
#define CV64(p) reinterpret_cast<const Vec<double>*>(p)

template <typename R, typename T> static inline R as_res(Res<T> r) {
    R out;
    out.result_code = r.result_code;
    out.vector = reinterpret_cast<decltype(out.vector)>(r.vector);
    return out;
}

#define BDSP_MATH_FACADE(S, T, VEC, CVEC, RES, HV)                                                                     \
    extern "C" RES sin##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_SIN, (T)0, false)); }                       \
    extern "C" RES cos##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_COS, (T)0, false)); }                       \
    extern "C" RES tan##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_TAN, (T)0, false)); }                       \
    extern "C" RES asin##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ASIN, (T)0, false)); }                     \
    extern "C" RES acos##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ACOS, (T)0, false)); }                     \
    extern "C" RES atan##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ATAN, (T)0, false)); }                     \
    extern "C" RES sinh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_SINH, (T)0, false)); }                     \
    extern "C" RES cosh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_COSH, (T)0, false)); }                     \
    extern "C" RES tanh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_TANH, (T)0, false)); }                     \
    extern "C" RES asinh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ASINH, (T)0, false)); }                   \
    extern "C" RES acosh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ACOSH, (T)0, false)); }                   \
    extern "C" RES atanh##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ATANH, (T)0, false)); }                   \
    extern "C" RES sqrt##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_SQRT, (T)0, false)); }                     \
    extern "C" RES square##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_SQUARE, (T)0, false)); }                 \
    extern "C" RES ln##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_LN, (T)0, false)); }                         \
    extern "C" RES exp##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_EXP, (T)0, false)); }                       \
    extern "C" RES abs##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_ABS, (T)0, true)); }                        \
    extern "C" RES root##S(HV* v, T degree) { return as_res<RES>(op_math<T>(VEC(v), M_POWF, (T)1 / degree, false)); }  \
    extern "C" RES bdsp_powf##S(HV* v, T e) { return as_res<RES>(op_math<T>(VEC(v), M_POWF, e, false)); }              \
    extern "C" RES log##S(HV* v, T base) { return as_res<RES>(op_math<T>(VEC(v), M_LOG, base, false)); }               \
    extern "C" RES bdsp_expf##S(HV* v, T base) { return as_res<RES>(op_math<T>(VEC(v), M_EXPF, base, false)); }        \
    extern "C" RES wrap##S(HV* v, T d) { return as_res<RES>(op_math<T>(VEC(v), M_WRAP, d, true)); }                    \
    extern "C" RES unwrap##S(HV* v, T d) { return as_res<RES>(op_unwrap<T>(VEC(v), d)); }                              \
    extern "C" RES ln_approx##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_LN, (T)0, true)); }                   \
    extern "C" RES exp_approx##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_EXP, (T)0, true)); }                 \
    extern "C" RES sin_approx##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_SIN, (T)0, true)); }                 \
    extern "C" RES cos_approx##S(HV* v) { return as_res<RES>(op_math<T>(VEC(v), M_COS, (T)0, true)); }                 \
    extern "C" RES log_approx##S(HV* v, T base) { return as_res<RES>(op_math<T>(VEC(v), M_LOG, base, true)); }         \
    extern "C" RES expf_approx##S(HV* v, T base) { return as_res<RES>(op_math<T>(VEC(v), M_EXPF, base, true)); }       \
    extern "C" RES powf_approx##S(HV* v, T e) { return as_res<RES>(op_math<T>(VEC(v), M_POWF, e, true)); }             \
    extern "C" RES diff##S(HV* v) { return as_res<RES>(op_diff<T>(VEC(v), false)); }                                   \
    extern "C" RES diff_with_start##S(HV* v) { return as_res<RES>(op_diff<T>(VEC(v), true)); }                         \
    extern "C" RES cum_sum##S(HV* v) { return as_res<RES>(op_cum_sum<T>(VEC(v))); }                                    \
    extern "C" RES add_smaller_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary_smaller<T>(VEC(v), CVEC(o), EW_ADD)); } \
    extern "C" RES sub_smaller_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary_smaller<T>(VEC(v), CVEC(o), EW_SUB)); } \
    extern "C" RES mul_smaller_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary_smaller<T>(VEC(v), CVEC(o), EW_MUL)); } \
    extern "C" RES div_smaller_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary_smaller<T>(VEC(v), CVEC(o), EW_DIV)); } \
    extern "C" int32_t get_real_imag##S(HV* v, HV* re, HV* im) { return op_get_real_imag<T>(VEC(v), VEC(re), VEC(im)); } \
    extern "C" RES set_real_imag##S(HV* v, const HV* re, const HV* im) { return as_res<RES>(op_set_pair<T>(VEC(v), CVEC(re), CVEC(im), false)); } \
    extern "C" RES set_mag_phase##S(HV* v, const HV* m, const HV* p) { return as_res<RES>(op_set_pair<T>(VEC(v), CVEC(m), CVEC(p), true)); } \
    extern "C" int32_t split_into##S(const HV* v, HV** targets, size_t len) { return op_split_into<T>(CVEC(v), reinterpret_cast<Vec<T>**>(targets), len); } \
    extern "C" RES merge##S(HV* v, HV* const* sources, size_t len) { return as_res<RES>(op_merge<T>(VEC(v), reinterpret_cast<Vec<T>* const*>(sources), len)); } \
    extern "C" RES interpolate_hermite##S(HV* v, T factor, T delay) { return as_res<RES>(op_interpolate_hermite<T>(VEC(v), factor, delay)); }

#define BDSP_FACADE(S, T, VEC, CVEC, RES, HV, CPLX, RFN, CFN)                                                         \
    extern "C" HV* new##S(int32_t is_complex, int32_t domain, T init_value, size_t length, T delta) {                  \
        return reinterpret_cast<HV*>(vec_new<T>(is_complex, domain, init_value, length, delta));                       \
    }                                                                                                                  \
    extern "C" HV* new_with_performance_options##S(int32_t is_complex, int32_t domain, T init_value, size_t length,    \
                                                   T delta, size_t) {                                                  \
        return reinterpret_cast<HV*>(vec_new<T>(is_complex, domain, init_value, length, delta));                       \
    }                                                                                                                  \
    extern "C" HV* new_with_detailed_performance_options##S(int32_t is_complex, int32_t domain, T init_value,          \
                                                            size_t length, T delta, size_t, size_t, size_t, size_t,    \
                                                            size_t) {                                                  \
        return reinterpret_cast<HV*>(vec_new<T>(is_complex, domain, init_value, length, delta));                       \
    }                                                                                                                  \
    extern "C" void delete_vector##S(HV* v) { vec_delete(VEC(v)); }                                                    \
    extern "C" HV* clone##S(HV* v) {                                                                                   \
        Vec<T>* s = VEC(v);                                                                                            \
        Vec<T>* c = vec_new<T>(s->is_complex, s->domain, (T)0, 0, s->delta);                                           \
        if (!c) return nullptr;                                                                                        \
        if (reserve(&c->d, &c->cap, s->len, false, 0) != 0) { vec_delete(c); return nullptr; }                          \
        if (s->len) cudaMemcpyAsync(c->d, s->d, s->len * sizeof(T), cudaMemcpyDeviceToDevice, g_stream);               \
        c->len = s->len;                                                                                               \
        return reinterpret_cast<HV*>(c);                                                                               \
    }                                                                                                                  \
    extern "C" T get_value##S(const HV* v, size_t index) {                                                             \
        T r = (T)NAN;                                                                                                  \
        if (index < CVEC(v)->len) {                                                                                    \
            cudaMemcpyAsync(&r, CVEC(v)->d + index, sizeof(T), cudaMemcpyDeviceToHost, g_stream);                      \
            cudaStreamSynchronize(g_stream);                                                                           \
        }                                                                                                              \
        return r;                                                                                                      \
    }                                                                                                                  \
    extern "C" void set_value##S(HV* v, size_t index, T value) {                                                       \
        if (index < VEC(v)->len) {                                                                                     \
            cudaMemcpyAsync(VEC(v)->d + index, &value, sizeof(T), cudaMemcpyHostToDevice, g_stream);                   \
            cudaStreamSynchronize(g_stream);                                                                           \
            VEC(v)->version++;                                                                                         \
        }                                                                                                              \
    }                                                                                                                  \
    extern "C" int32_t is_complex##S(const HV* v) { return CVEC(v)->is_complex ? 1 : 0; }                              \
    extern "C" int32_t get_domain##S(const HV* v) { return CVEC(v)->domain; }                                          \
    extern "C" size_t get_len##S(const HV* v) { return CVEC(v)->len; }                                                 \
    extern "C" void set_len##S(HV* v, size_t len) { (void)vec_resize(VEC(v), len); }                                   \
    extern "C" size_t get_points##S(const HV* v) { return points_of(CVEC(v)); }                                        \
    extern "C" T get_delta##S(const HV* v) { return CVEC(v)->delta; }                                                  \
    extern "C" const T* data##S(const HV* v) { return host_mirror(CVEC(v)); }                                          \
    extern "C" const CPLX* complex_data##S(const HV* v) { return reinterpret_cast<const CPLX*>(host_mirror(CVEC(v))); } \
    extern "C" size_t get_allocated_len##S(const HV* v) { return CVEC(v)->cap; }                                       \
    extern "C" RES overwrite_data##S(HV* v, const T* data, size_t len) {                                               \
        Vec<T>* s = VEC(v);                                                                                            \
        int code = E_ARG_LEN;                                                                                          \
        if (len < s->len) { /* strict, as in the reference (Q9) */                                                     \
            code = 0;                                                                                                  \
            if (len) {                                                                                                 \
                cudaMemcpyAsync(s->d, data, len * sizeof(T), cudaMemcpyHostToDevice, g_stream);                        \
                cudaStreamSynchronize(g_stream);                                                                       \
            }                                                                                                          \
            s->version++;                                                                                              \
        }                                                                                                              \
        RES r; r.result_code = code; r.vector = v; return r;                                                           \
    }                                                                                                                  \
    extern "C" RES add##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_ADD)); }              \
    extern "C" RES sub##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_SUB)); }              \
    extern "C" RES div##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_DIV)); }              \
    extern "C" RES mul##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_MUL)); }              \
    extern "C" RES add_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_ADD)); }       \
    extern "C" RES sub_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_SUB)); }       \
    extern "C" RES div_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_DIV)); }       \
    extern "C" RES mul_vector##S(HV* v, const HV* o) { return as_res<RES>(op_binary(VEC(v), CVEC(o), EW_MUL)); }       \
    extern "C" RES real_offset##S(HV* v, T c) { return as_res<RES>(op_real_const(VEC(v), EW_OFFSET, c)); }             \
    extern "C" RES real_scale##S(HV* v, T c) { return as_res<RES>(op_real_const(VEC(v), EW_SCALE, c)); }               \
    extern "C" RES complex_offset##S(HV* v, T re, T im) { return as_res<RES>(op_complex_const(VEC(v), EW_OFFSET, re, im)); } \
    extern "C" RES complex_scale##S(HV* v, T re, T im) { return as_res<RES>(op_complex_const(VEC(v), EW_SCALE, re, im)); } \
    extern "C" RES complex_divide##S(HV* v, T re, T im) { return as_res<RES>(op_complex_divide(VEC(v), re, im)); }     \
    extern "C" RES conj##S(HV* v) { return as_res<RES>(op_complex_const(VEC(v), EW_CONJ, (T)0, (T)0)); }               \
    extern "C" RES to_complex##S(HV* v) { return as_res<RES>(op_to_complex(VEC(v))); }                                 \
    extern "C" RES magnitude##S(HV* v) { return as_res<RES>(op_c2r(VEC(v), C2R_MAG_SQRT)); }                           \
    extern "C" RES magnitude_squared##S(HV* v) { return as_res<RES>(op_c2r(VEC(v), C2R_MAG_SQ)); }                     \
    extern "C" RES phase##S(HV* v) { return as_res<RES>(op_c2r(VEC(v), C2R_PHASE)); }                                  \
    extern "C" RES to_real##S(HV* v) { return as_res<RES>(op_c2r(VEC(v), C2R_REAL)); }                                 \
    extern "C" RES to_imag##S(HV* v) { return as_res<RES>(op_c2r(VEC(v), C2R_IMAG)); }                                 \
    extern "C" int32_t get_magnitude##S(HV* v, HV* d) { return op_get_c2r(VEC(v), VEC(d), C2R_MAG_SQRT); }             \
    extern "C" int32_t get_magnitude_squared##S(HV* v, HV* d) { return op_get_c2r(VEC(v), VEC(d), C2R_MAG_SQ); }       \
    extern "C" int32_t get_phase##S(HV* v, HV* d) { return op_get_c2r(VEC(v), VEC(d), C2R_PHASE); }                    \
    extern "C" int32_t get_real##S(HV* v, HV* d) { return op_get_c2r(VEC(v), VEC(d), C2R_REAL); }                      \
    extern "C" int32_t get_imag##S(HV* v, HV* d) { return op_get_c2r(VEC(v), VEC(d), C2R_IMAG); }                      \
    extern "C" int32_t get_mag_phase##S(HV* v, HV* m, HV* p) { return op_get_mag_phase(VEC(v), VEC(m), VEC(p)); }      \
    extern "C" RES plain_fft##S(HV* v) { return as_res<RES>(op_fft(VEC(v), false, false, false)); }                    \
    extern "C" RES plain_ifft##S(HV* v) { return as_res<RES>(op_fft(VEC(v), true, false, false)); }                    \
    extern "C" RES fft##S(HV* v) { return as_res<RES>(op_fft(VEC(v), false, true, false)); }                           \
    extern "C" RES ifft##S(HV* v) { return as_res<RES>(op_fft(VEC(v), true, true, false)); }                           \
    extern "C" RES bdsp_fft_magnitude##S(HV* v) { return as_res<RES>(op_fft(VEC(v), false, true, true)); }             \
    extern "C" RES swap_halves##S(HV* v) { return as_res<RES>(op_rotate(VEC(v), true)); }                              \
    extern "C" RES fft_shift##S(HV* v) { return as_res<RES>(op_rotate(VEC(v), true)); }                                \
    extern "C" RES ifft_shift##S(HV* v) { return as_res<RES>(op_rotate(VEC(v), false)); }                              \
    extern "C" RES zero_pad##S(HV* v, size_t points, int32_t opt) { return as_res<RES>(op_zero_pad(VEC(v), points, opt)); } \
    extern "C" RES zero_interleave##S(HV* v, int32_t factor) { return as_res<RES>(op_zero_interleave(VEC(v), factor)); } \
    extern "C" RES convolve_signal##S(HV* v, const HV* h) {                                                            \
        return as_res<RES>(op_convolve_signal(VEC(v), const_cast<Vec<T>*>(CVEC(h))));                                  \
    }                                                                                                                  \
    extern "C" RES convolve##S(HV* v, int32_t kind, T rolloff, T ratio, size_t len) {                                  \
        RealFn<T> f; f.kind = kind == 0 ? 0 : 1; f.rolloff = rolloff;                                                  \
        return as_res<RES>(op_convolve_fn<T>(VEC(v), f, ratio, len));                                         \
    }                                                                                                                  \
    extern "C" RES convolve_real##S(HV* v, RFN fn, const void* data, uint8_t, T ratio, size_t len) {                   \
        RealFn<T> f; f.fn = fn; f.data = data;                                                                         \
        return as_res<RES>(op_convolve_fn<T>(VEC(v), f, ratio, len));                                         \
    }                                                                                                                  \
    extern "C" RES convolve_complex##S(HV* v, CFN fn, const void* data, uint8_t, T ratio, size_t len) {                \
        return as_res<RES>(op_convolve_cfn<T, CPLX>(VEC(v), fn, data, ratio, len));                                    \
    }                                                                                                                  \
    extern "C" RES multiply_frequency_response##S(HV* v, int32_t kind, T rolloff, T ratio) {                           \
        RealFn<T> f; f.kind = kind == 0 ? 0 : 1; f.rolloff = rolloff;                                                  \
        return as_res<RES>(op_mul_freq_resp<T>(VEC(v), f, ratio));                                                     \
    }                                                                                                                  \
    extern "C" RES multiply_frequency_response_real##S(HV* v, RFN fn, const void* data, uint8_t, T ratio) {            \
        RealFn<T> f; f.fn = fn; f.data = data;                                                                         \
        return as_res<RES>(op_mul_freq_resp<T>(VEC(v), f, ratio));                                                     \
    }                                                                                                                  \
    extern "C" RES multiply_frequency_response_complex##S(HV* v, CFN fn, const void* data, uint8_t, T ratio) {         \
        return as_res<RES>(op_mul_freq_resp_c<T, CPLX>(VEC(v), fn, data, ratio));                                      \
    }                                                                                                                  \
    extern "C" RES interpolatef##S(HV* v, int32_t kind, T rolloff, T factor, T delay, size_t len) {                    \
        RealFn<T> f; f.kind = kind == 0 ? 0 : 1; f.rolloff = rolloff;                                                  \
        return as_res<RES>(op_interpolatef<T>(VEC(v), f, factor, delay, len));                                         \
    }                                                                                                                  \
    extern "C" RES interpolatef_custom##S(HV* v, RFN fn, const void* data, uint8_t, T factor, T delay, size_t len) {   \
        RealFn<T> f; f.fn = fn; f.data = data;                                                                         \
        return as_res<RES>(op_interpolatef<T>(VEC(v), f, factor, delay, len));                                         \
    }                                                                                                                  \
    extern "C" RES interpolate_lin##S(HV* v, T factor, T delay) { return as_res<RES>(op_interpolate_lin(VEC(v), factor, delay)); } \
    extern "C" RES interpolatei##S(HV* v, int32_t kind, T rolloff, int32_t factor) {                                  \
        RealFn<T> f; f.kind = kind == 0 ? 0 : 1; f.rolloff = rolloff;                                                  \
        return as_res<RES>(op_interpolatei<T>(VEC(v), f, true, (uint32_t)factor));                                     \
    }                                                                                                                  \
    extern "C" RES interpolatei_custom##S(HV* v, RFN fn, const void* data, uint8_t is_symmetric, int32_t factor) {     \
        RealFn<T> f; f.fn = fn; f.data = data;                                                                         \
        return as_res<RES>(op_interpolatei<T>(VEC(v), f, is_symmetric != 0, (uint32_t)factor));                        \
    }                                                                                                                  \
    extern "C" RES interpolate##S(HV* v, int32_t kind, T rolloff, size_t dest_points, T delay) {                       \
        RealFn<T> f; f.kind = kind == 0 ? 0 : 1; f.rolloff = rolloff;                                                  \
        return as_res<RES>(op_interpolate<T>(VEC(v), &f, true, dest_points, delay));                                   \
    }                                                                                                                  \
    extern "C" RES interpolate_custom##S(HV* v, RFN fn, const void* data, uint8_t is_symmetric, size_t dest_points, T delay) { \
        RealFn<T> f; f.fn = fn; f.data = data;                                                                         \
        return as_res<RES>(op_interpolate<T>(VEC(v), &f, is_symmetric != 0, dest_points, delay));                      \
    }                                                                                                                  \
    extern "C" RES interpft##S(HV* v, size_t dest_points) { return as_res<RES>(op_interpolate<T>(VEC(v), nullptr, true, dest_points, (T)0)); } \
    extern "C" RES multiply_complex_exponential##S(HV* v, T a, T b) { return as_res<RES>(op_mul_cexp(VEC(v), a, b)); } \
    extern "C" RES mirror##S(HV* v) { return as_res<RES>(op_mirror(VEC(v))); }                                         \
    extern "C" RES plain_sfft##S(HV* v) { return as_res<RES>(op_sfft<T>(VEC(v), false, nullptr)); }                    \
    extern "C" RES sfft##S(HV* v) { return as_res<RES>(op_sfft<T>(VEC(v), true, nullptr)); }                           \
    extern "C" RES windowed_sfft##S(HV* v, int32_t k) { WinFn<T> w; w.kind = k; return as_res<RES>(op_sfft<T>(VEC(v), true, &w)); } \
    extern "C" RES plain_sifft##S(HV* v) { return as_res<RES>(op_sifft<T>(VEC(v), false, nullptr)); }                  \
    extern "C" RES sifft##S(HV* v) { return as_res<RES>(op_sifft<T>(VEC(v), true, nullptr)); }                         \
    extern "C" RES windowed_sifft##S(HV* v, int32_t k) { WinFn<T> w; w.kind = k; return as_res<RES>(op_sifft<T>(VEC(v), true, &w)); } \
    extern "C" RES apply_custom_window##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                              \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_window_fn<T>(VEC(v), w, false)); } \
    extern "C" RES unapply_custom_window##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                            \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_window_fn<T>(VEC(v), w, true)); } \
    extern "C" RES windowed_custom_fft##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                              \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_windowed_fft_fn<T>(VEC(v), w)); } \
    extern "C" RES windowed_custom_ifft##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                             \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_windowed_ifft_fn<T>(VEC(v), w)); } \
    extern "C" RES windowed_custom_sfft##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                             \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_sfft<T>(VEC(v), true, &w)); } \
    extern "C" RES windowed_custom_sifft##S(HV* v, BdspWindowFn##S fn, const void* data, uint8_t sym) {                            \
        WinFn<T> w; w.fn = fn; w.data = data; w.symmetric = sym != 0; return as_res<RES>(op_sifft<T>(VEC(v), true, &w)); } \
    extern "C" RES map_inplace_real##S(HV* v, T (*map)(T, size_t)) { return as_res<RES>(op_map_inplace_real<T>(VEC(v), map)); } \
    extern "C" RES map_inplace_complex##S(HV* v, CPLX (*map)(CPLX, size_t)) { return as_res<RES>(op_map_inplace_complex<T, CPLX>(VEC(v), map)); } \
    extern "C" BdspPointerResult map_aggregate_real##S(const HV* v, const void* (*map)(T, size_t), const void* (*aggr)(const void*, const void*)) { \
        return op_map_aggregate<T, T>(CVEC(v), false, map, aggr); }                                                    \
    extern "C" BdspPointerResult map_aggregate_complex##S(const HV* v, const void* (*map)(CPLX, size_t), const void* (*aggr)(const void*, const void*)) { \
        return op_map_aggregate<T, CPLX>(CVEC(v), true, map, aggr); }                                                  \
    BDSP_MATH_FACADE(S, T, VEC, CVEC, RES, HV)                                                                         \
    extern "C" RES apply_window##S(HV* v, int32_t w) { return as_res<RES>(op_window(VEC(v), w, false)); }              \
    extern "C" RES unapply_window##S(HV* v, int32_t w) { return as_res<RES>(op_window(VEC(v), w, true)); }             \
    extern "C" RES windowed_fft##S(HV* v, int32_t w) { return as_res<RES>(op_windowed_fft(VEC(v), w)); }               \
    extern "C" RES windowed_ifft##S(HV* v, int32_t w) { return as_res<RES>(op_windowed_ifft(VEC(v), w)); }             \
    extern "C" RES prepare_argument##S(HV* v) { return as_res<RES>(op_prepare_argument(VEC(v), false)); }              \
    extern "C" RES prepare_argument_padded##S(HV* v) { return as_res<RES>(op_prepare_argument(VEC(v), true)); }        \
    extern "C" RES correlate##S(HV* v, const HV* o) { return as_res<RES>(op_correlate(VEC(v), CVEC(o))); }             \
    extern "C" RES reverse##S(HV* v) { return as_res<RES>(op_reverse(VEC(v))); }                                       \
    extern "C" RES decimatei##S(HV* v, uint32_t f, uint32_t d) { return as_res<RES>(op_decimatei(VEC(v), f, d)); }     \
    extern "C" int32_t bdsp_upload##S(HV* v, const T* host, size_t len) { return upload(VEC(v), host, len); }          \
    extern "C" int32_t bdsp_download##S(const HV* v, T* host, size_t len) { return download(CVEC(v), host, len, true); } \
    extern "C" int32_t bdsp_download_async##S(const HV* v, T* host, size_t len) { return download(CVEC(v), host, len, false); } \
    /* mutable access: caches derived from the vector's contents (the overlap-save plan) are invalidated */             \
    extern "C" void* bdsp_device_ptr##S(HV* v) { VEC(v)->version++; return VEC(v)->d; }                                \
    extern "C" int32_t bdsp_scale_mul_mag_phase##S(HV* v, T cre, T cim, const HV* w, HV* m, HV* p, int32_t wb) {       \
        return scale_mul_mag_phase<T>(VEC(v), cre, cim, CVEC(w), VEC(m), VEC(p), wb);                                  \
    }

BDSP_FACADE(32, float, V32, CV32, BdspVecResult32, BdspVec32, BdspComplex32, BdspRealFn32, BdspComplexFn32)
BDSP_FACADE(64, double, V64, CV64, BdspVecResult64, BdspVec64, BdspComplex64, BdspRealFn64, BdspComplexFn64)


// ---- reductions (facade32.rs:193-321, 848-931; facade64.rs likewise) ---------------------------------
#define BDSP_REDUCE_FACADE(S, T, TP, CVEC, CPLX, CPLXP, HV)                                                            \
    extern "C" BdspScalarResult##S real_dot_product##S(const HV* v, const HV* o) {                                     \
        double r[2]; BdspScalarResult##S out; out.result_code = dot_of<T>(CVEC(v), CVEC(o), false, 0, r);              \
        out.result = out.result_code ? (T)0 : (T)r[0]; if (!out.result_code && erroneous(CVEC(v))) out.result_code = -1; return out; } \
    extern "C" BdspScalarResult##S real_dot_product_prec##S(const HV* v, const HV* o) {                                \
        double r[2]; BdspScalarResult##S out; out.result_code = dot_of<T>(CVEC(v), CVEC(o), false, 1, r);              \
        out.result = out.result_code ? (T)0 : (T)r[0]; if (!out.result_code && erroneous(CVEC(v))) out.result_code = -1; return out; } \
    extern "C" BdspComplexScalarResult##S complex_dot_product##S(const HV* v, const HV* o) {                           \
        double r[2]; BdspComplexScalarResult##S out; out.result_code = dot_of<T>(CVEC(v), CVEC(o), true, 0, r);        \
        out.result.re = out.result_code ? (T)0 : (T)r[0]; out.result.im = out.result_code ? (T)0 : (T)r[1];            \
        if (!out.result_code && erroneous(CVEC(v))) out.result_code = -1; return out; }                                \
    extern "C" BdspComplexScalarResult##S complex_dot_product_prec##S(const HV* v, const HV* o) {                      \
        double r[2]; BdspComplexScalarResult##S out; out.result_code = dot_of<T>(CVEC(v), CVEC(o), true, 1, r);        \
        out.result.re = out.result_code ? (T)0 : (T)r[0]; out.result.im = out.result_code ? (T)0 : (T)r[1];            \
        if (!out.result_code && erroneous(CVEC(v))) out.result_code = -1; return out; }                                \
    extern "C" T real_sum##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 0, r); return (T)r[0]; }                  \
    extern "C" T real_sum_sq##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 0, r); return (T)r[2]; }               \
    extern "C" CPLX complex_sum##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 0, r); CPLX c; c.re = (T)r[0]; c.im = (T)r[1]; return c; } \
    extern "C" CPLX complex_sum_sq##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 0, r); CPLX c; c.re = (T)r[2]; c.im = (T)r[3]; return c; } \
    extern "C" TP real_sum_prec##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 1, r); return (TP)r[0]; }           \
    extern "C" TP real_sum_sq_prec##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 1, r); return (TP)r[2]; }        \
    extern "C" CPLXP complex_sum_prec##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 1, r); CPLXP c; c.re = (TP)r[0]; c.im = (TP)r[1]; return c; } \
    extern "C" CPLXP complex_sum_sq_prec##S(const HV* v) { double r[4]; sums_of<T>(CVEC(v), 1, r); CPLXP c; c.re = (TP)r[2]; c.im = (TP)r[3]; return c; } \
    extern "C" BdspStatistics##S real_statistics##S(const HV* v) {                                                     \
        StatsRaw raw; BdspStatistics##S out; stats_of<T>(CVEC(v), 1, 0, &raw); stats_fill_real(&out, raw); return out; } \
    extern "C" BdspComplexStatistics##S complex_statistics##S(const HV* v) {                                           \
        StatsRaw raw; BdspComplexStatistics##S out; stats_of<T>(CVEC(v), 1, 0, &raw); stats_fill_complex<BdspComplexStatistics##S, T>(&out, raw); return out; } \
    extern "C" BdspStatistics64 real_statistics_prec##S(const HV* v) {                                                 \
        StatsRaw raw; BdspStatistics64 out; stats_of<T>(CVEC(v), 1, 1, &raw); stats_fill_real(&out, raw); return out; } \
    extern "C" BdspComplexStatistics64 complex_statistics_prec##S(const HV* v) {                                       \
        StatsRaw raw; BdspComplexStatistics64 out; stats_of<T>(CVEC(v), 1, 1, &raw); stats_fill_complex<BdspComplexStatistics64, double>(&out, raw); return out; } \
    extern "C" int32_t real_statistics_split##S(const HV* v, BdspStatistics##S* data, size_t len) {                    \
        if (len == 0) return 0; if (len > 16) return E_ARG_LEN;                                                        \
        StatsRaw raw[16]; int rc = stats_of<T>(CVEC(v), (int)len, 0, raw); if (rc) return rc;                          \
        for (size_t i = 0; i < len; i++) stats_fill_real(&data[i], raw[i]); return 0; }                                \
    extern "C" int32_t complex_statistics_split##S(const HV* v, BdspComplexStatistics##S* data, size_t len) {          \
        if (len == 0) return 0; if (len > 16) return E_ARG_LEN;                                                        \
        StatsRaw raw[16]; int rc = stats_of<T>(CVEC(v), (int)len, 0, raw); if (rc) return rc;                          \
        for (size_t i = 0; i < len; i++) stats_fill_complex<BdspComplexStatistics##S, T>(&data[i], raw[i]); return 0; } \
    extern "C" int32_t real_statistics_split_prec##S(const HV* v, BdspStatistics64* data, size_t len) {                \
        if (len == 0) return 0; if (len > 16) return E_ARG_LEN;                                                        \
        StatsRaw raw[16]; int rc = stats_of<T>(CVEC(v), (int)len, 1, raw); if (rc) return rc;                          \
        for (size_t i = 0; i < len; i++) stats_fill_real(&data[i], raw[i]); return 0; }                                \
    extern "C" int32_t complex_statistics_split_prec##S(const HV* v, BdspComplexStatistics64* data, size_t len) {      \
        if (len == 0) return 0; if (len > 16) return E_ARG_LEN;                                                        \
        StatsRaw raw[16]; int rc = stats_of<T>(CVEC(v), (int)len, 1, raw); if (rc) return rc;                          \
        for (size_t i = 0; i < len; i++) stats_fill_complex<BdspComplexStatistics64, double>(&data[i], raw[i]); return 0; }

BDSP_REDUCE_FACADE(32, float, double, CV32, BdspComplex32, BdspComplex64, BdspVec32)
BDSP_REDUCE_FACADE(64, double, double, CV64, BdspComplex64, BdspComplex64, BdspVec64)

extern "C" const char* bdsp_version(void) { return "basic_dsp_b200 0.1.0 (sm_100a)"; }
extern "C" const char* bdsp_last_error(void) { return get_last_error(); }
extern "C" int32_t bdsp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
extern "C" int32_t bdsp_set_device(int32_t device) { BDSP_CUDA_OK(cudaSetDevice(device)); return 0; }
extern "C" int32_t bdsp_sync(void) { BDSP_CUDA_OK(cudaStreamSynchronize(g_stream)); return 0; }
extern "C" void bdsp_set_stream(void* s) { g_stream = reinterpret_cast<cudaStream_t>(s); workspace_bind_stream(g_stream); }
extern "C" void* bdsp_stream_create(void) {
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    return s;
}
extern "C" void bdsp_stream_destroy(void* s) {
    if (!s) return;
    cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(s));
    workspace_release_stream(reinterpret_cast<cudaStream_t>(s));
    cudaStreamDestroy(reinterpret_cast<cudaStream_t>(s));
}
extern "C" int32_t bdsp_stream_sync(void* s) { BDSP_CUDA_OK(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(s))); return 0; }

extern "C" int32_t bdsp_fft_rows_c32(const void* in, void* out, size_t points, size_t rows, int32_t flags) { return fft_rows<float>(in, out, points, rows, flags); }
extern "C" int32_t bdsp_fft_rows_c64(const void* in, void* out, size_t points, size_t rows, int32_t flags) { return fft_rows<double>(in, out, points, rows, flags); }
extern "C" int32_t bdsp_fft_frames_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return fft_frames<float>(in, out, points, hop, frames, flags);
}
extern "C" int32_t bdsp_fft_frames_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return fft_frames<double>(in, out, points, hop, frames, flags);
}
extern "C" int32_t bdsp_ifft_frames_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return ifft_frames<float>(in, out, points, hop, frames, flags);
}
extern "C" int32_t bdsp_ifft_frames_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return ifft_frames<double>(in, out, points, hop, frames, flags);
}
extern "C" int32_t bdsp_welch_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags, float fs) {
    return welch<float>(in, out, points, hop, frames, flags, (double)fs);
}
extern "C" int32_t bdsp_welch_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags, double fs) {
    return welch<double>(in, out, points, hop, frames, flags, fs);
}
extern "C" int32_t bdsp_csd_c32(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags, float fs) {
    return cross_spectrum<float>(x, y, out, points, hop, frames, flags, (double)fs, false);
}
extern "C" int32_t bdsp_csd_c64(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags, double fs) {
    return cross_spectrum<double>(x, y, out, points, hop, frames, flags, fs, false);
}
extern "C" int32_t bdsp_coherence_c32(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return cross_spectrum<float>(x, y, out, points, hop, frames, flags, 1.0, true);
}
extern "C" int32_t bdsp_coherence_c64(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags) {
    return cross_spectrum<double>(x, y, out, points, hop, frames, flags, 1.0, true);
}
extern "C" BdspConvPlan* bdsp_conv_plan_create_c32(const void* h, size_t L) { return reinterpret_cast<BdspConvPlan*>(conv_plan_create<float>(h, L)); }
extern "C" BdspConvPlan* bdsp_conv_plan_create_c64(const void* h, size_t L) { return reinterpret_cast<BdspConvPlan*>(conv_plan_create<double>(h, L)); }
extern "C" void bdsp_conv_plan_destroy(BdspConvPlan* plan) {
    ConvPlan* p = reinterpret_cast<ConvPlan*>(plan);
    if (!p) return;
    cudaStreamSynchronize(g_stream);
    if (p->ols) ols_plan_destroy(p->ols);
    if (p->taps) cudaFree(p->taps);
    delete p;
}
extern "C" int32_t bdsp_convolve_signal_rows_c32(const void* in, void* out, size_t points, size_t rows, const BdspConvPlan* plan) {
    return conv_rows<float>(in, out, points, rows, reinterpret_cast<const ConvPlan*>(plan));
}
extern "C" int32_t bdsp_convolve_signal_rows_c64(const void* in, void* out, size_t points, size_t rows, const BdspConvPlan* plan) {
    return conv_rows<double>(in, out, points, rows, reinterpret_cast<const ConvPlan*>(plan));
}
#define BDSP_ROWS(S, T)                                                                                                          \
    extern "C" int32_t bdsp_magnitude_rows_c##S(const void* in, void* out, size_t points, size_t rows) {                              \
        return c2r_rows<T>(C2R_MAG_HYPOT, in, out, points, rows);                                                                     \
    }                                                                                                                                 \
    extern "C" int32_t bdsp_magnitude_squared_rows_c##S(const void* in, void* out, size_t points, size_t rows) {                      \
        return c2r_rows<T>(C2R_MAG_SQ, in, out, points, rows);                                                                        \
    }                                                                                                                                 \
    extern "C" int32_t bdsp_phase_rows_c##S(const void* in, void* out, size_t points, size_t rows) {                                  \
        return c2r_rows<T>(C2R_PHASE, in, out, points, rows);                                                                         \
    }                                                                                                                                 \
    extern "C" int32_t bdsp_scale_mul_mag_phase_rows_c##S(void* v, const void* w, void* magnitude, void* phase, size_t points,        \
                                                          size_t rows, T scale_re, T scale_im, int32_t write_back) {                  \
        return chain_rows<T>(v, w, magnitude, phase, points, rows, scale_re, scale_im, write_back);                                   \
    }                                                                                                                                 \
    extern "C" int32_t bdsp_interpolatef_rows##S(const void* in, void* out, size_t points, size_t rows, int32_t is_complex,           \
                                                 int32_t impulse_response, T rolloff, T interpolation_factor, T delay, size_t len,    \
                                                 size_t* new_points) {                                                                \
        return interp_rows<T>(in, out, points, rows, is_complex, impulse_response, rolloff, interpolation_factor, delay, len,         \
                              new_points);                                                                                            \
    }
BDSP_ROWS(32, float)
BDSP_ROWS(64, double)
#undef BDSP_ROWS

extern "C" void* bdsp_malloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) { set_last_error("bdsp_malloc(%zu) failed", bytes); return nullptr; }
    return p;
}
extern "C" void bdsp_free(void* p) { if (p) { cudaStreamSynchronize(g_stream); cudaFree(p); } }
extern "C" size_t bdsp_mem_free(void) {
    size_t f = 0, t = 0;
    return cudaMemGetInfo(&f, &t) == cudaSuccess ? f : 0;
}
extern "C" void* bdsp_malloc_host(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { set_last_error("bdsp_malloc_host(%zu) failed", bytes); return nullptr; }
    return p;
}
extern "C" void bdsp_free_host(void* p) { if (p) cudaFreeHost(p); }
extern "C" int32_t bdsp_memcpy_h2d(void* d, const void* h, size_t bytes) { BDSP_CUDA_OK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, g_stream)); return 0; }
extern "C" int32_t bdsp_memcpy_d2h(void* h, const void* d, size_t bytes) { BDSP_CUDA_OK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, g_stream)); return 0; }
extern "C" int32_t bdsp_memset(void* d, int32_t value, size_t bytes) { BDSP_CUDA_OK(cudaMemsetAsync(d, value, bytes, g_stream)); return 0; }
extern "C" void* bdsp_event_create(void) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    return e;
}
extern "C" void bdsp_event_destroy(void* e) { if (e) cudaEventDestroy(reinterpret_cast<cudaEvent_t>(e)); }
extern "C" int32_t bdsp_event_record(void* e) { BDSP_CUDA_OK(cudaEventRecord(reinterpret_cast<cudaEvent_t>(e), g_stream)); return 0; }
extern "C" float bdsp_event_elapsed_ms(void* a, void* b) {
    float ms = -1.f;
    if (cudaEventSynchronize(reinterpret_cast<cudaEvent_t>(b)) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, reinterpret_cast<cudaEvent_t>(a), reinterpret_cast<cudaEvent_t>(b)) != cudaSuccess) return -1.f;
    return ms;
}
extern "C" uint64_t bdsp_kernel_launch_count(void) { return launch_count(); }
