// libgl_commit: context, stage orchestration and the extern "C" boundary declared in include/gl_commit.h.
//
// Host-side mirror of plonky2 fri/oracle.rs · PolynomialBatch::from_values / from_coeffs, hash/merkle_tree.rs ·
// MerkleTree::new and fri/prover.rs · fri_committed_trees (driven from /root/reference/src/p3/mod.rs:250,260).
// Everything here is plumbing around the kernels in ntt.cuh / merkle.cuh / fri.cuh; there is no CPU compute path.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges cost nothing unless a profiler injects the NVTX library

#include <cstdio>
#include <algorithm>
#include <exception>
#include <cstring>
#include <cstdlib>
#include <condition_variable>
#include <map>
#include <thread>
#include <utility>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "../../include/gl_commit.h"
#include "fri.cuh"
#include "gates.cuh"
#include "merkle.cuh"
#include "microbench.cuh"
#include "ntt.cuh"
#include "ntt2.cuh"
#include "openings.cuh"
#include "peer_sync.cuh"
#include "permutation.cuh"

#ifndef LEAF_BLOCK
#define LEAF_BLOCK 128   // threads per CTA of the leaf-hash kernels (tests/variants.py builds other sizes)
#endif

namespace {

struct GlError {
    int code;
    std::string msg;
};

// NVTX ranges named after plonky2's own TimingTree labels (fri/oracle.rs · from_values / from_coeffs: "IFFT", "FFT + blinding",
// "transpose LDEs", "build Merkle tree"; fri/prover.rs: "fold codewords in the commitment phase", "find proof-of-work witness"), so a
// timeline of the drop-in reads like upstream's `timing` output.  Host-side ranges around the enqueue of each stage.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};


#define GL_THROW(code, ...)                              \
    do {                                                 \
        char _b[512];                                    \
        snprintf(_b, sizeof _b, __VA_ARGS__);            \
        throw GlError{code, _b};                         \
    } while (0)

#define CUDA_CHECK(expr)                                                                                   \
    do {                                                                                                   \
        cudaError_t _e = (expr);                                                                           \
        if (_e != cudaSuccess) {                                                                           \
            int _c = (_e == cudaErrorMemoryAllocation) ? GL_ERR_OOM : GL_ERR_CUDA;                         \
            GL_THROW(_c, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);      \
        }                                                                                                  \
    } while (0)

// Device allocations are recycled through a small per-process free list: a commit needs ~11 GB of leaves/digests at
// 2^20 x 135 and cudaMalloc/cudaFree of that size is milliseconds of driver time per call.  Exact-size reuse only.
struct DevPool {
    std::mutex mu;
    std::multimap<std::pair<int, size_t>, uint64_t*> free_list;   // (device, words) -> pointer
    size_t cached_words = 0;
    static DevPool& get() { static DevPool p; return p; }
    uint64_t* take(int dev, size_t words) {
        std::lock_guard<std::mutex> lk(mu);
        auto it = free_list.find({dev, words});
        if (it == free_list.end()) return nullptr;
        uint64_t* p = it->second;
        free_list.erase(it);
        cached_words -= words;
        return p;
    }
    void give(int dev, size_t words, uint64_t* p) {
        std::lock_guard<std::mutex> lk(mu);
        free_list.insert({{dev, words}, p});
        cached_words += words;
    }
    void trim(int dev) {   // release everything cached for `dev` (on allocation failure / context destruction)
        std::lock_guard<std::mutex> lk(mu);
        for (auto it = free_list.begin(); it != free_list.end();) {
            if (it->first.first == dev) { cudaFree(it->second); cached_words -= it->first.second; it = free_list.erase(it); }
            else ++it;
        }
    }
};

struct DevBuf {
    uint64_t* p = nullptr;
    size_t words = 0;
    int dev = -1;
    void ensure(size_t w) {
        if (w <= words) return;
        release();
        if (w == 0) w = 1;
        CUDA_CHECK(cudaGetDevice(&dev));
        p = DevPool::get().take(dev, w);
        if (!p) {
            cudaError_t e = cudaMalloc(&p, w * sizeof(uint64_t));
            if (e == cudaErrorMemoryAllocation) {   // give cached blocks back to the driver and retry once
                cudaGetLastError();
                DevPool::get().trim(dev);
                e = cudaMalloc(&p, w * sizeof(uint64_t));
            }
            if (e != cudaSuccess) { p = nullptr; CUDA_CHECK(e); }
        }
        words = w;
    }
    void release() {
        // Released while an error unwinds the call: kernels or copies enqueued before the failure may still be touching the
        // buffer, and the pool is shared with other contexts — wait for the device before handing it on (error path only).
        if (p && std::uncaught_exceptions() > 0) cudaDeviceSynchronize();
        if (p) DevPool::get().give(dev, words, p);
        p = nullptr;
        words = 0;
    }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
};

inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }
inline uint32_t log2_exact(uint64_t n) {
    uint32_t l = 0;
    while ((1ULL << l) < n) l++;
    return l;
}
inline uint32_t h_bitrev(uint32_t x, uint32_t bits) {
    uint32_t r = 0;
    for (uint32_t i = 0; i < bits; i++) { r = (r << 1) | (x & 1); x >>= 1; }
    return r;
}

// how the log_n stages are split into shared-memory passes (each <= 10 stages, as even as possible)
std::vector<uint32_t> plan_passes(uint32_t n, uint32_t max_a = 10) {
    std::vector<uint32_t> v;
    if (n < 3) return v;
    uint32_t k = (n + max_a - 1) / max_a, base = n / k, rem = n % k;
    for (uint32_t i = 0; i < k; i++) v.push_back(base + (i < rem ? 1 : 0));
    return v;
}

struct CosetTable {   // pre-scale factors g^j, j < N, fused into the first pass's loads
    uint64_t g = 1;
    DevBuf F;
};

struct Tree {
    uint64_t n_leaves = 0;
    uint32_t leaf_len = 0, pitch = 0, cap_height = 0, degree_log = 0, rate_bits = 0;
    DevBuf leaves, digests, coeffs, d_cap;
    bool has_coeffs = false;
    std::vector<uint64_t> cap;
    // leaves [n_leaves][pitch], digests, cap on the device and on the host; the coefficients are the caller's
    Tree(uint64_t n_leaves_, uint32_t leaf_len_, uint32_t pitch_, uint32_t cap_height_)
        : n_leaves(n_leaves_), leaf_len(leaf_len_), pitch(pitch_), cap_height(cap_height_), cap(4ULL << cap_height_) {
        leaves.ensure(n_leaves * pitch);
        digests.ensure(n_digests() * 4);
        d_cap.ensure(4ULL << cap_height);
    }
    uint64_t n_digests() const { return 2 * (n_leaves - (1ULL << cap_height)); }
};

struct Fri {
    uint64_t len = 0;
    uint32_t rate_bits = 0, cap_height = 0;
    uint64_t shift = gl::COSET_SHIFT;
    uint32_t last_arity_bits = 0;
    DevBuf coeffs, values, tmp;   // values are kept in bit-reversed order (what the next layer's leaves need)
    Fri(uint64_t len_, uint32_t rate_bits_, uint32_t cap_height_) : len(len_), rate_bits(rate_bits_), cap_height(cap_height_) {
        coeffs.ensure(2 * len); values.ensure(2 * len); tmp.ensure(2 * len);
    }
};

struct Quotient {
    gl_handle wires = 0;
    uint64_t n_rows = 0;
    uint32_t n_challenges = 0;
    DevBuf acc, powers;
};

struct Openings {
    uint32_t log_n = 0;
    DevBuf final_poly, comp, refs, pw;   // final_poly / composition: N extension elements each
};

// The objects of one kind a context hands out.  All kinds draw their handles from the context's one counter, so a handle of one kind is
// never valid as another.
template <class T>
struct Handles {
    const char* kind;   // in "unknown <kind> handle"
    std::map<gl_handle, std::unique_ptr<T>> live;
    gl_handle put(gl_ctx* c, std::unique_ptr<T> obj);
    T* get(gl_handle h) const;
    void drop(gl_ctx* c, gl_handle h);   // waits for the context's stream: enqueued work may still use the object's buffers
};

}  // namespace

struct gl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string err;
    std::map<uint32_t, std::unique_ptr<DevBuf>> roots;                       // log_n -> W
    std::map<uint32_t, std::unique_ptr<DevBuf>> pass_roots;                  // a -> w_{2^a}^e, e < 7*2^a/8 (round twiddles)
    std::map<uint64_t, std::unique_ptr<std::vector<CosetTable>>> lde_tables;  // (log_n, rate_bits) -> per coset
    std::map<std::pair<uint64_t, uint32_t>, std::unique_ptr<CosetTable>> coset_cache;   // (shift, log_len) -> g^j: FRI layers / final-poly LDE
    size_t coset_cache_words = 0;
    DevBuf in_stage, vals, scratch, hash_state;
    Handles<Tree> trees{"tree"};
    Handles<Fri> fris{"fri"};
    Handles<Openings> openings{"openings"};
    Handles<Quotient> quotients{"quotient"};
    float aux_ms = 0;
    gl_handle next_handle = 1;
    cudaStream_t copy_stream = nullptr;   // host->device column copies of gl_commit, overlapped with the NTTs
    // multi-GPU exchange of gl_*_lde_scatter (DESIGN.md §6 has the measurements): cosets owned by this rank are stored by the NTT
    // itself (no copy); the others stay local in send_buf and the COPY ENGINES ship them on send_stream (one strided 2-D peer copy per
    // owner segment) while the next coset's NTT runs — no SM time, no NVLink stalls inside the NTT
    cudaStream_t send_stream = nullptr;
    cudaStream_t pull_stream = nullptr;   // peer -> local coefficient pulls of the coset-sharded plan.  NOT the copy stream: a stream that has
                                          // carried peer copies keeps its copy-engine binding, and host->device chunks queued behind it then
                                          // serialise with the send stream's shipments (measured: an 8 ms stall of the first shipment)
    cudaEvent_t ev_ntt[2] = {}, ev_sent[2] = {};
    bool sent_pending[2] = {false, false};
    DevBuf send_buf[2];
    std::set<const uint64_t*> own_ipc;    // buffers exported by gl_dev_ipc_alloc (to tell the local leaf buffer from mapped peers)
    bool trace = false;                    // GL_TRACE=1: per-coset timeline of the overlapped exchange on stderr (development aid)
    std::vector<cudaEvent_t> trace_ev;     // base, then per coset: ntt start, ntt end, send start, send end
    cudaEvent_t ev_sync = nullptr, ev_copyback = nullptr;
    std::vector<cudaEvent_t> chunk_ev, pull_ev, own_ev;
    DevBuf sync_err;                      // error word of the streamed coset plan's ticket waits (peer_sync.cuh)
    cudaEvent_t ev[GL_N_STAGES + 1] = {};
    float stage_ms[GL_N_STAGES] = {};
    uint32_t launches[GL_N_STAGES] = {};
    int sm_count = 148;
};

namespace {

template <class T>
gl_handle Handles<T>::put(gl_ctx* c, std::unique_ptr<T> obj) {
    const gl_handle h = c->next_handle++;
    live[h] = std::move(obj);
    return h;
}
template <class T>
T* Handles<T>::get(gl_handle h) const {
    auto it = live.find(h);
    if (it == live.end()) GL_THROW(GL_ERR_HANDLE, "unknown %s handle %llu", kind, (unsigned long long)h);
    return it->second.get();
}
template <class T>
void Handles<T>::drop(gl_ctx* c, gl_handle h) {
    get(h);
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    live.erase(h);
}

const uint64_t* get_roots(gl_ctx* c, uint32_t log_n) {
    auto it = c->roots.find(log_n);
    if (it != c->roots.end()) return it->second->p;
    size_t half = log_n ? (size_t)1 << (log_n - 1) : 1;
    std::vector<uint64_t> w(half);
    uint64_t root = gl::h_root_of_unity(log_n), cur = 1;
    for (size_t e = 0; e < half; e++) { w[e] = cur; cur = gl::h_mul(cur, root); }
    auto buf = std::make_unique<DevBuf>();
    buf->ensure(half);
    CUDA_CHECK(cudaMemcpyAsync(buf->p, w.data(), half * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    const uint64_t* p = buf->p;
    c->roots[log_n] = std::move(buf);
    return p;
}

const uint64_t* get_pass_roots(gl_ctx* c, uint32_t a) {
    auto it = c->pass_roots.find(a);
    if (it != c->pass_roots.end()) return it->second->p;
    const size_t T = (size_t)1 << a, n = T;   // the full circle: radix-16 rounds reach exponents up to 15T/16
    std::vector<uint64_t> w(n ? n : 1);
    uint64_t root = gl::h_root_of_unity(a), cur = 1;
    for (size_t e = 0; e < n; e++) {
        w[e] = e < (T >> 1) ? cur : gl::P - w[e - (T >> 1)];   // w_T^(e) = -w_T^(e - T/2); never 0, so P - x is canonical
        cur = gl::h_mul(cur, root);
    }
    auto buf = std::make_unique<DevBuf>();
    buf->ensure(w.size());
    CUDA_CHECK(cudaMemcpyAsync(buf->p, w.data(), w.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    const uint64_t* p = buf->p;
    c->pass_roots[a] = std::move(buf);
    return p;
}

// F[j] = g^j, j < 2^log_n, filled ON THE DEVICE (square-and-multiply over the 32 host-computed g^(2^k)): no O(N) host loop, no
// H2D copy and no stream synchronisation in the per-call paths (gl_fri_fold, gl_openings_lde)
void fill_coset_table(gl_ctx* c, CosetTable& t, uint64_t g, uint32_t log_n) {
    t.g = g;
    if (log_n < 3) return;   // ntt_tiny_kernel takes g itself
    ntt::PowTable pt{};
    uint64_t sq = gl::canon(g);
    for (uint32_t k = 0; k < 32; k++) { pt.g2k[k] = sq; sq = gl::h_mul(sq, sq); }
    const uint64_t n = 1ULL << log_n;
    t.F.ensure(n);
    ntt::powers_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, c->stream>>>(t.F.p, n, pt);
    CUDA_CHECK(cudaGetLastError());
}

// pre-scale table of a single coset NTT (the FRI layers re-evaluate on shift^arity; prove_openings on shift 7), kept per context:
// a prover that proves repeatedly hits the cache; bounded at 2^25 words (256 MB)
const CosetTable* get_coset_table(gl_ctx* c, uint64_t g, uint32_t log_len) {
    auto key = std::make_pair(g, log_len);
    auto it = c->coset_cache.find(key);
    if (it != c->coset_cache.end()) return it->second.get();
    const size_t words = (size_t)1 << log_len;
    if (c->coset_cache_words + words > ((size_t)1 << 25)) {
        CUDA_CHECK(cudaStreamSynchronize(c->stream));   // a cached table may still be read by an enqueued pass
        c->coset_cache.clear();
        c->coset_cache_words = 0;
    }
    auto t = std::make_unique<CosetTable>();
    fill_coset_table(c, *t, g, log_len);
    c->coset_cache_words += words;
    const CosetTable* p = t.get();
    c->coset_cache[key] = std::move(t);
    return p;
}

// coset s of the LDE evaluates at 7 * w_R^s * w_N^m
const std::vector<CosetTable>& get_lde_tables(gl_ctx* c, uint32_t log_n, uint32_t rate_bits) {
    uint64_t key = ((uint64_t)log_n << 32) | rate_bits;
    auto it = c->lde_tables.find(key);
    if (it != c->lde_tables.end()) return *it->second;
    auto v = std::make_unique<std::vector<CosetTable>>((size_t)1 << rate_bits);
    uint64_t wR = gl::h_root_of_unity(log_n + rate_bits), g = gl::COSET_SHIFT;
    for (uint32_t s = 0; s < (1u << rate_bits); s++) {
        fill_coset_table(c, (*v)[s], g, log_n);
        g = gl::h_mul(g, wR);
    }
    auto& ref = *v;
    c->lde_tables[key] = std::move(v);
    return ref;
}

template <int G, int A>
void launch_pass_a(gl_ctx* c, const ntt::PassParams& p, uint32_t threads, size_t smem, uint32_t grid) {   // smem <= 44 KB for every (G, a)
    ntt::ntt_pass_kernel<G, A><<<grid, threads, smem, c->stream>>>(p);
}
// second-generation pass (ntt2.cuh): two columns per thread, carry-save butterflies, all-shift radix-16 last round
// once per device: the shared-memory opt-in of a second-generation pass kernel (the attribute belongs to the function on a device)
template <int G, int A>
void prepare_pass2() {
    constexpr size_t smem = ntt2::smem_words<A, G>() * 8;
    if (smem > 48 * 1024) {
        static std::once_flag once[64];
        int dev = 0;
        CUDA_CHECK(cudaGetDevice(&dev));
        cudaError_t e = cudaSuccess;
        std::call_once(once[dev & 63], [&] { e = cudaFuncSetAttribute(ntt2::ntt_pass_kernel<G, A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
        CUDA_CHECK(e);
    }
}
template <int G, int A>
void launch_pass2_a(gl_ctx* c, const ntt::PassParams& p, uint32_t grid) {
    constexpr size_t smem = ntt2::smem_words<A, G>() * 8;
    constexpr uint32_t threads = (1u << A) * G / 16;
    prepare_pass2<G, A>();
    ntt2::ntt_pass_kernel<G, A><<<grid, threads, smem, c->stream>>>(p);
}

// Loads every kernel the streamed coset plan launches into the current device's context (CUDA loads functions lazily, at their first
// launch, and a load may have to synchronise the context while the runtime's lock is held).  The plan parks ticket waits on the GPU: a
// first launch that happens while such a wait spins would block behind it — holding the lock another thread of the process needs to launch
// the very signal the wait is spinning for (observed with gl_commit_multi on two devices: every wait ran into its time limit).  So nothing
// may be loaded after the first wait is enqueued.
template <int G, int A>
void preload_pass2() {
    cudaFuncAttributes at;
    CUDA_CHECK(cudaFuncGetAttributes(&at, ntt2::ntt_pass_kernel<G, A>));
    prepare_pass2<G, A>();
    if constexpr (A > 3) preload_pass2<G, A - 1>();
}
void preload_stream_kernels() {
    static std::once_flag once[64];
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    cudaError_t e = cudaSuccess;
    std::call_once(once[dev & 63], [&] {
        cudaFuncAttributes at;
        auto load = [&](const void* f) { if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, f); };
        load((const void*)ntt::transpose_in_kernel);
        load((const void*)ntt::ntt_tiny_kernel);
        load((const void*)peersync::signal_kernel);
        load((const void*)peersync::wait_kernel);
        load((const void*)merkle::leaf_absorb_kernel<LEAF_BLOCK>);
        load((const void*)merkle::tree_level_kernel<128>);
    });
    CUDA_CHECK(e);
    preload_pass2<4, 10>();
    preload_pass2<8, 10>();
}
template <int G>
void launch_pass2(gl_ctx* c, ntt::PassParams p, uint32_t cols_padded, uint32_t* launches) {
    p.ncg = cols_padded / G;
    const uint64_t grid = (uint64_t)p.ncg << (p.log_n - p.a);
    if (grid >= (1ULL << 31)) GL_THROW(GL_ERR_UNSUPPORTED, "NTT grid too large");
    switch (p.a) {
        case 3: launch_pass2_a<G, 3>(c, p, (uint32_t)grid); break;
        case 4: launch_pass2_a<G, 4>(c, p, (uint32_t)grid); break;
        case 5: launch_pass2_a<G, 5>(c, p, (uint32_t)grid); break;
        case 6: launch_pass2_a<G, 6>(c, p, (uint32_t)grid); break;
        case 7: launch_pass2_a<G, 7>(c, p, (uint32_t)grid); break;
        case 8: launch_pass2_a<G, 8>(c, p, (uint32_t)grid); break;
        case 9: launch_pass2_a<G, 9>(c, p, (uint32_t)grid); break;
        case 10: launch_pass2_a<G, 10>(c, p, (uint32_t)grid); break;
        default: GL_THROW(GL_ERR_INVALID, "run_ntt: pass size %u has no second-generation kernel", p.a);
    }
    CUDA_CHECK(cudaGetLastError());
    if (launches) (*launches)++;
}

// first-generation pass (ntt.cuh): instantiated for what run_ntt launches with it — <2,0>, <4,3..10> and <8,3..9>
template <int G>
void launch_pass(gl_ctx* c, ntt::PassParams p, uint32_t cols_padded, uint32_t* launches) {
    p.ncg = cols_padded / G;
    uint32_t T = 1u << p.a;
    uint32_t threads = T * G / 8;
    size_t smem = ((size_t)(T + (T >> 3)) * G + (T - (T >> 3))) * 8;   // padded tile + 7T/8 twiddles
    uint64_t grid = (uint64_t)p.ncg << (p.log_n - p.a);
    if (grid >= (1ULL << 31)) GL_THROW(GL_ERR_UNSUPPORTED, "NTT grid too large");
    if constexpr (G == 2) {
        launch_pass_a<G, 0>(c, p, threads, smem, (uint32_t)grid);      // FRI matrices: generic pass size
    } else {
        switch (p.a) {                                                  // pass size as a compile-time constant
            case 3: launch_pass_a<G, 3>(c, p, threads, smem, (uint32_t)grid); break;
            case 4: launch_pass_a<G, 4>(c, p, threads, smem, (uint32_t)grid); break;
            case 5: launch_pass_a<G, 5>(c, p, threads, smem, (uint32_t)grid); break;
            case 6: launch_pass_a<G, 6>(c, p, threads, smem, (uint32_t)grid); break;
            case 7: launch_pass_a<G, 7>(c, p, threads, smem, (uint32_t)grid); break;
            case 8: launch_pass_a<G, 8>(c, p, threads, smem, (uint32_t)grid); break;
            case 9: launch_pass_a<G, 9>(c, p, threads, smem, (uint32_t)grid); break;
            case 10:
                if constexpr (G == 4) { launch_pass_a<G, 10>(c, p, threads, smem, (uint32_t)grid); break; }
                [[fallthrough]];                                        // 8 columns: run_ntt takes 10-stage passes in 4-column tiles
            default: GL_THROW(GL_ERR_INVALID, "bad pass size %u", p.a);
        }
    }
    CUDA_CHECK(cudaGetLastError());
    if (launches) (*launches)++;
}

// Batched NTT of `cols_padded` columns (multiple of G) of a row-major matrix.
//   forward (ifft=false): src -> dst in in-place-DIF order (row p = X[bitrev(p)]), optional coset pre-scale `pre`;
//                         later passes run in place on dst.
//   ifft:                 all passes but the last run IN PLACE ON src (destroyed); last pass stores to dst in natural
//                         coefficient order scaled by 1/N.
//   scatter != nullptr (forward only): the last pass stores to the leaf owners (store_mode 2); dst is then only the
//                         scratch the earlier passes work in.
void run_ntt(gl_ctx* c, uint64_t* src, uint32_t src_pitch, uint64_t* dst, uint32_t dst_pitch, uint32_t cols_padded,
             uint32_t log_n, bool ifft, const CosetTable* pre, int G, uint32_t* launches, const ntt::Scatter* scatter = nullptr,
             const uint64_t* const* src_list = nullptr) {
    // src_list (forward, second-generation kernel only): the cols_padded / G column groups are read from separate [N][G] blocks
    // src_list[cg] (src and src_pitch ignored); the later passes run in place on dst with 8-column tiles when the width allows
    if (src_list && (ifft || scatter || (G != 4 && G != 8) || log_n < 3 || cols_padded / G > (uint32_t)ntt::MAX_PEERS))
        GL_THROW(GL_ERR_INVALID, "run_ntt: unsupported multi-source transform");
    const uint64_t* W = get_roots(c, log_n);
    uint64_t n_inv = ifft ? gl::h_inv(((uint64_t)1 << log_n) % gl::P) : 1;
    auto passes = plan_passes(log_n, 10);
    if (passes.empty()) {
        dim3 grid((cols_padded + 63) / 64, 1u << log_n);
        ntt::ntt_tiny_kernel<<<grid, 64, 0, c->stream>>>(src, dst, src_pitch, dst_pitch, cols_padded, log_n,
                                                         gl::h_root_of_unity(log_n), pre ? pre->g : 1, scatter ? 2 : (ifft ? 1 : 0), n_inv,
                                                         scatter ? *scatter : ntt::Scatter{});
        CUDA_CHECK(cudaGetLastError());
        if (launches) (*launches)++;
        return;
    }
    uint32_t log_blk = log_n;
    for (size_t i = 0; i < passes.size(); i++) {
        bool first = i == 0, last = i + 1 == passes.size();
        ntt::PassParams p{};
        p.log_n = log_n;
        p.log_blk = log_blk;
        p.a = passes[i];
        p.W = W;
        p.Wa = get_pass_roots(c, passes[i]);
        p.pre = (first && pre) ? pre->F.p : nullptr;
        p.store_mode = (ifft && last) ? 1 : 0;
        p.scale = (ifft && last) ? n_inv : 1;
        if (scatter && last) {
            p.store_mode = 2;
            memcpy(p.peer, scatter->peer, sizeof p.peer);
            p.scatter_row0 = scatter->row0; p.log_rows_per_peer = scatter->log_rows_per_peer;
            p.scatter_col0 = scatter->col0; p.scatter_pitch = scatter->pitch; p.scatter_ncols = scatter->ncols;
        }
        if (ifft) {
            p.src = src; p.src_pitch = src_pitch;
            p.dst = last ? dst : src; p.dst_pitch = last ? dst_pitch : src_pitch;
        } else {
            p.src = first ? src : dst; p.src_pitch = first ? src_pitch : dst_pitch;
            p.dst = dst; p.dst_pitch = dst_pitch;
        }
        // 128-bit accesses need even pitches and 16-byte aligned bases (true for every buffer this library lays out)
        const bool aligned = p.src_pitch % 2 == 0 && p.dst_pitch % 2 == 0 && ((uintptr_t)p.src % 16 == 0) && ((uintptr_t)p.dst % 16 == 0);
        if (src_list) {
            int g = G;
            if (first) {
                p.src_list = 1; p.src = nullptr; p.src_pitch = (uint32_t)G;
                for (uint32_t k = 0; k < cols_padded / G; k++) {
                    if ((uintptr_t)src_list[k] % 16) GL_THROW(GL_ERR_INVALID, "run_ntt: misaligned source block");
                    p.peer[k] = const_cast<uint64_t*>(src_list[k]);
                }
            } else if (cols_padded % 8 == 0) {
                g = 8;
            }
            if (p.dst_pitch % 2 || (uintptr_t)p.dst % 16) GL_THROW(GL_ERR_INVALID, "run_ntt: misaligned destination");
            g == 8 ? launch_pass2<8>(c, p, cols_padded, launches) : launch_pass2<4>(c, p, cols_padded, launches);
        } else if ((G == 8 || G == 4) && aligned) {
            G == 8 ? launch_pass2<8>(c, p, cols_padded, launches) : launch_pass2<4>(c, p, cols_padded, launches);
        } else {
            // first-generation kernel: the 2-column FRI matrices, and column groups whose base or pitch is not 16-byte aligned
            switch (G) {
                case 8:   // a 10-stage pass in 4-column tiles keeps 512 threads / 40 KB shared memory per CTA
                    p.a == 10 ? launch_pass<4>(c, p, cols_padded, launches) : launch_pass<8>(c, p, cols_padded, launches);
                    break;
                case 4: launch_pass<4>(c, p, cols_padded, launches); break;
                case 2: launch_pass<2>(c, p, cols_padded, launches); break;
                default: GL_THROW(GL_ERR_INVALID, "bad column group");
            }
        }
        log_blk -= passes[i];
    }
}

// the tree above the leaf digests: layers 1..log_sub, one launch per layer
void merkle_levels(gl_ctx* c, uint64_t n_leaves, uint32_t cap_height, uint64_t* d_digests, uint64_t* d_cap, uint32_t* tree_launches) {
    const uint32_t log_sub = log2_exact(n_leaves) - cap_height;
    for (uint32_t layer = 1; layer <= log_sub; layer++) {
        uint64_t n_nodes = n_leaves >> layer;
        constexpr int TB = 128;
        merkle::tree_level_kernel<TB><<<(uint32_t)((n_nodes + TB - 1) / TB), TB, 0, c->stream>>>(d_digests, d_cap, layer, log_sub, n_nodes);
        CUDA_CHECK(cudaGetLastError());
        if (tree_launches) (*tree_launches)++;
    }
}

void merkle_build(gl_ctx* c, const uint64_t* d_leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t pitch,
                  uint32_t cap_height, uint64_t* d_digests, uint64_t* d_cap, uint32_t* leaf_launches,
                  uint32_t* tree_launches, cudaEvent_t after_leaves) {
    NvtxRange nv("build Merkle tree");
    uint32_t log_leaves = log2_exact(n_leaves);
    uint32_t log_sub = log_leaves - cap_height;
    constexpr int LB = LEAF_BLOCK;
    merkle::leaf_hash_kernel<LB><<<(uint32_t)((n_leaves + LB - 1) / LB), LB, 0, c->stream>>>(
        d_leaves, pitch, leaf_len, n_leaves, log_sub, d_digests, d_cap);
    CUDA_CHECK(cudaGetLastError());
    if (leaf_launches) (*leaf_launches)++;
    if (after_leaves) CUDA_CHECK(cudaEventRecord(after_leaves, c->stream));
    merkle_levels(c, n_leaves, cap_height, d_digests, d_cap, tree_launches);
}

// streaming leaf sponge (merkle.cuh · leaf_absorb_kernel): columns [col0, col1) of every leaf
void leaf_absorb(gl_ctx* c, const uint64_t* d_leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t pitch, uint32_t cap_height, uint32_t col0,
                 uint32_t col1, uint64_t* d_state, uint64_t* d_digests, uint64_t* d_cap, bool first, bool last, uint32_t* leaf_launches) {
    const uint32_t log_sub = log2_exact(n_leaves) - cap_height;
    constexpr int LB = LEAF_BLOCK;
    merkle::leaf_absorb_kernel<LB><<<(uint32_t)((n_leaves + LB - 1) / LB), LB, 0, c->stream>>>(d_leaves, pitch, leaf_len, col0, col1, n_leaves, log_sub,
                                                                                             d_state, d_digests, d_cap, first ? 1 : 0, last ? 1 : 0);
    CUDA_CHECK(cudaGetLastError());
    if (leaf_launches) (*leaf_launches)++;
}

void check_shape(uint32_t n_cols, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height) {
    if (n_cols == 0) GL_THROW(GL_ERR_INVALID, "empty polynomial batch");
    if (log_n + rate_bits > 31) GL_THROW(GL_ERR_UNSUPPORTED, "log_n + rate_bits = %u > 31", log_n + rate_bits);
    if (cap_height > log_n + rate_bits)
        GL_THROW(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len()) (cap_height=%u, log2(leaves)=%u)",
                 cap_height, log_n + rate_bits);
}

// The end of a tree built on the compute stream: digests (if asked for) and cap to the host, and a handle (if asked for)
void finish_tree(gl_ctx* c, std::unique_ptr<Tree> t, uint64_t* out_digests, uint64_t* out_cap, gl_handle* out_tree) {
    CUDA_CHECK(cudaMemcpyAsync(t->cap.data(), t->d_cap.p, t->cap.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    if (out_digests && t->n_digests())
        CUDA_CHECK(cudaMemcpyAsync(out_digests, t->digests.p, t->n_digests() * 32, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    memcpy(out_cap, t->cap.data(), t->cap.size() * 8);
    if (out_tree) *out_tree = c->trees.put(c, std::move(t));
}

void copy_row(gl_ctx* c, const Tree* t, uint64_t row, uint64_t* out_row) {
    CUDA_CHECK(cudaMemcpyAsync(out_row, t->leaves.p + row * t->pitch, (size_t)t->leaf_len * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
}

void record(gl_ctx* c, int i) { CUDA_CHECK(cudaEventRecord(c->ev[i], c->stream)); }

// Stage clock of one call: stage i runs from event i to event i + 1.  reset_stages zeroes the launch counts and times of the stages
// [first, end) the call books; read_stages waits for the call's work and reads their times.
void reset_stages(gl_ctx* c, int first, int end) {
    for (int i = first; i < end; i++) { c->launches[i] = 0; c->stage_ms[i] = 0; }
}
void read_stages(gl_ctx* c, int first, int end) {
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    for (int i = first; i < end; i++) CUDA_CHECK(cudaEventElapsedTime(&c->stage_ms[i], c->ev[i], c->ev[i + 1]));
}

void ensure_events(std::vector<cudaEvent_t>& v, size_t n) {   // at least n events without timing
    while (v.size() < n) {
        v.push_back(nullptr);
        CUDA_CHECK(cudaEventCreateWithFlags(&v.back(), cudaEventDisableTiming));
    }
}

// Column groups of 8 words (64 B row segments); a shard whose padding to 8 would waste >= 4 columns runs in groups of 4 (32 B = one
// sector) instead.  coeff_pitch is the row pitch the shard's coefficients are laid out with.
int column_group(uint32_t n_cols, uint32_t coeff_pitch) {
    if (coeff_pitch % 4 || coeff_pitch < n_cols) GL_THROW(GL_ERR_INVALID, "coeff_pitch must be a multiple of 4 and >= n_cols");
    const int G = (round_up(n_cols, 8) - n_cols >= 4) ? 4 : 8;
    if (coeff_pitch < round_up(n_cols, (uint32_t)G)) GL_THROW(GL_ERR_INVALID, "coeff_pitch too small for the padded column group");
    return G;
}

// Transpose of `n_cols` device columns (column-major, col_stride apart) into columns [0, width) of the row-major [N][pitch] `coeffs`
// (zero beyond n_cols).  Values (vals != nullptr) go through the [N][pitch] scratch `vals` and an iNTT of groups of G columns.
// split_events: the call is one stage clock of its own (the transpose ends the transpose stage, the iNTT the iNTT stage).
void intt_columns(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t width, uint32_t log_n,
                  uint64_t* vals, uint64_t* coeffs, uint32_t pitch, int G, bool split_events) {
    const uint64_t N = 1ULL << log_n;
    dim3 tb(32, 8), tg((uint32_t)((N + 31) / 32), (width + 31) / 32);
    ntt::transpose_in_kernel<<<tg, tb, 0, c->stream>>>(d_cols, col_stride, vals ? vals : coeffs, pitch, width, n_cols, N);
    CUDA_CHECK(cudaGetLastError());
    c->launches[GL_STAGE_TRANSPOSE]++;
    if (split_events) record(c, GL_STAGE_INTT);
    if (vals) run_ntt(c, vals, pitch, coeffs, pitch, round_up(n_cols, (uint32_t)G), log_n, true, nullptr, G, &c->launches[GL_STAGE_INTT]);
    if (split_events) record(c, GL_STAGE_LDE);
}

// One coset of a scattered LDE whose rows belong (partly) to other ranks: the coset is evaluated into send_buf[b] and the copy
// engines ship it on send_stream, one strided 2-D peer copy per owner segment (no SM time), while the next coset's NTT runs on the
// compute stream.  The buffer is reused only after its previous shipment has finished.
void ship_coset(gl_ctx* c, uint64_t* coeffs, uint32_t coeff_pitch, uint32_t cols_padded, uint32_t log_n, const CosetTable* tab, int G,
                const ntt::Scatter& sc, uint32_t col0, uint32_t row_pitch, int b) {
    const uint64_t N = 1ULL << log_n;
    uint64_t* buf = c->send_buf[b].p + col0;
    if (c->sent_pending[b]) CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->ev_sent[b], 0));
    auto mark = [&](cudaStream_t st) {
        if (!c->trace) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); c->trace_ev.push_back(e);
    };
    if (c->trace && c->trace_ev.empty()) mark(c->stream);
    mark(c->stream);
    run_ntt(c, coeffs, coeff_pitch, buf, row_pitch, cols_padded, log_n, false, tab, G, &c->launches[GL_STAGE_LDE]);
    mark(c->stream);
    CUDA_CHECK(cudaEventRecord(c->ev_ntt[b], c->stream));
    CUDA_CHECK(cudaStreamWaitEvent(c->send_stream, c->ev_ntt[b], 0));
    mark(c->send_stream);
    const uint64_t rpp = 1ULL << sc.log_rows_per_peer;
    for (uint64_t r = 0; r < N;) {
        const uint64_t grow = sc.row0 + r, owner = grow >> sc.log_rows_per_peer, lrow = grow & (rpp - 1);
        const uint64_t cnt = std::min<uint64_t>(N - r, rpp - lrow);
        CUDA_CHECK(cudaMemcpy2DAsync(sc.peer[owner] + lrow * sc.pitch + sc.col0, (size_t)sc.pitch * 8, buf + r * row_pitch,
                                     (size_t)row_pitch * 8, (size_t)sc.ncols * 8, cnt, cudaMemcpyDefault, c->send_stream));
        r += cnt;
    }
    mark(c->send_stream);
    c->launches[GL_STAGE_LDE]++;   // the shipment books as one launch of the LDE stage
    CUDA_CHECK(cudaEventRecord(c->ev_sent[b], c->send_stream));
    c->sent_pending[b] = true;
}

// iNTT + coset LDE of `n_cols` device columns (column-major, col_stride apart) into columns [col0, col0 + padded) of the
// row-major outputs.  Column groups are independent, so a batch can be processed in chunks (pipelined behind the
// host->device copies in gl_commit).  col0 must be a multiple of 8.
// scatter != nullptr: every coset's rows go to their owners' leaf buffers (d_rows is then the NTT scratch of one coset): a coset
// whose rows all belong to this rank is stored there by the NTT itself, every other coset is shipped by ship_coset.
void lde_columns(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t col0, uint32_t n_cols, uint32_t width,
                 uint32_t log_n, uint32_t rate_bits, int is_coeffs, uint64_t* d_vals, uint64_t* d_coeffs, uint32_t coeff_pitch,
                 uint64_t* d_rows, uint32_t row_pitch, int G, bool split_events, const ntt::Scatter* scatter = nullptr,
                 uint32_t first_coset = 0) {
    const uint64_t N = 1ULL << log_n;
    const uint32_t cols_padded = round_up(n_cols, G);
    NvtxRange nv_lde(is_coeffs ? "FFT + blinding (coset LDE, leaves stored bit-reversed: includes 'transpose LDEs')"
                               : "IFFT, FFT + blinding (coset LDE, leaves stored bit-reversed: includes 'transpose LDEs')");
    uint64_t* coeffs = d_coeffs + col0;
    intt_columns(c, d_cols, col_stride, n_cols, width, log_n, is_coeffs ? nullptr : d_vals + col0, coeffs, coeff_pitch, G, split_events);
    const auto& tabs = get_lde_tables(c, log_n, rate_bits);
    for (uint32_t k = 0; k < (1u << rate_bits); k++) {
        const uint32_t s = (k + first_coset) & ((1u << rate_bits) - 1);
        if (!scatter) {
            uint64_t* dst = d_rows + (uint64_t)h_bitrev(s, rate_bits) * N * row_pitch + col0;
            run_ntt(c, coeffs, coeff_pitch, dst, row_pitch, cols_padded, log_n, false, &tabs[s], G, &c->launches[GL_STAGE_LDE]);
            continue;
        }
        ntt::Scatter sc = *scatter;
        sc.row0 = (uint64_t)h_bitrev(s, rate_bits) * N;
        sc.col0 = scatter->col0 + col0;   // this chunk's columns inside the leaf row
        sc.ncols = n_cols;
        const bool all_local = scatter->self < ntt::MAX_PEERS && (sc.row0 >> sc.log_rows_per_peer) == scatter->self &&
                               ((sc.row0 + N - 1) >> sc.log_rows_per_peer) == scatter->self;
        if (all_local)
            run_ntt(c, coeffs, coeff_pitch, d_rows + col0, row_pitch, cols_padded, log_n, false, &tabs[s], G, &c->launches[GL_STAGE_LDE], &sc);
        else
            ship_coset(c, coeffs, coeff_pitch, cols_padded, log_n, &tabs[s], G, sc, col0, row_pitch, (int)(k & 1));
    }
}

void lde_stage(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
               int is_coeffs, uint64_t* d_coeffs, uint32_t coeff_pitch, uint64_t* d_rows, uint32_t row_pitch) {
    const int G = column_group(n_cols, coeff_pitch);
    if (!is_coeffs) c->vals.ensure(((uint64_t)1 << log_n) * coeff_pitch);
    lde_columns(c, d_cols, col_stride, 0, n_cols, coeff_pitch, log_n, rate_bits, is_coeffs, c->vals.p, d_coeffs, coeff_pitch, d_rows,
                row_pitch, G, true);
}

// Host columns -> c->in_stage in chunks on the copy stream; fn(c0, nc, first) runs on the compute stream once chunk
// [c0, c0 + nc) has landed, i.e. transpose + iNTT + LDE of chunk k overlap the PCIe copy of chunk k+1 (column groups are
// independent polynomials).  Chunks grow 8, 16, 24, 24, ... columns: only the small first copy is exposed.  Chunk offsets
// are multiples of 8.  With pinned host memory the copies overlap completely.
template <class F>
void for_each_host_chunk(gl_ctx* c, const uint64_t* const* host_cols, uint32_t n_cols, uint64_t N, F&& fn, bool doubling = false) {
    for (uint32_t j = 0; j < n_cols; j++)
        if (!host_cols[j]) GL_THROW(GL_ERR_INVALID, "cols[%u] is NULL", j);
    c->in_stage.ensure(N * n_cols);
    std::vector<std::pair<uint32_t, uint32_t>> chunks;
    // 8, 16, 24, 24, ... columns; `doubling` (the caller also hashes each chunk, so compute per chunk dwarfs its copy): 8, 16, 32, 64, 64, ...
    // — fewer, larger launches and fewer sponge-state hand-overs
    for (uint32_t c0 = 0, sz = 8; c0 < n_cols; c0 += sz, sz = doubling ? std::min(2 * sz, 64u) : std::min(sz + 8, 24u))
        chunks.push_back({c0, std::min(sz, n_cols - c0)});
    ensure_events(c->chunk_ev, chunks.size());
    CUDA_CHECK(cudaEventRecord(c->ev_sync, c->stream));              // in_stage may still be read by an earlier call
    CUDA_CHECK(cudaStreamWaitEvent(c->copy_stream, c->ev_sync, 0));
    for (size_t k = 0; k < chunks.size(); k++) {
        for (uint32_t j = chunks[k].first; j < chunks[k].first + chunks[k].second; j++)
            CUDA_CHECK(cudaMemcpyAsync(c->in_stage.p + (uint64_t)j * N, host_cols[j], N * 8, cudaMemcpyHostToDevice, c->copy_stream));
        CUDA_CHECK(cudaEventRecord(c->chunk_ev[k], c->copy_stream));
    }
    for (size_t k = 0; k < chunks.size(); k++) {
        CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->chunk_ev[k], 0));
        fn(chunks[k].first, chunks[k].second, k == 0);
    }
}

int commit_impl(gl_ctx* c, const uint64_t* const* host_cols, const uint64_t* d_cols_in, uint64_t col_stride, uint32_t n_cols,
                uint32_t log_n, uint32_t rate_bits, uint32_t cap_height, int is_coeffs, uint64_t* out_coeffs,
                uint64_t* out_leaves, uint64_t* out_digests, uint64_t* out_cap, gl_handle* out_batch) {
    check_shape(n_cols, log_n, rate_bits, cap_height);
    if (!out_cap) GL_THROW(GL_ERR_INVALID, "out_cap is NULL");
    const uint64_t N = 1ULL << log_n, R = N << rate_bits;
    const uint32_t pitch = round_up(n_cols, 8);
    // warm the tables before the timed region starts
    get_roots(c, log_n);
    get_lde_tables(c, log_n, rate_bits);
    auto t = std::make_unique<Tree>(R, n_cols, pitch, cap_height);
    t->degree_log = log_n; t->rate_bits = rate_bits; t->has_coeffs = true;
    t->coeffs.ensure(N * pitch);
    reset_stages(c, 0, GL_N_STAGES);

    record(c, GL_STAGE_H2D);
    // Host columns with more than one chunk: the leaf sponge runs chunk by chunk behind the LDE of each chunk (leaf_absorb_kernel), so the
    // PCIe copy of the later chunks hides behind hashing; the stage clock then books those launches under "lde" (they interleave with it).
    const bool hash_per_chunk = host_cols && n_cols > 8;
    bool leaves_hashed = false;
    if (host_cols) {
        if (!is_coeffs) c->vals.ensure(N * pitch);
        if (hash_per_chunk) c->hash_state.ensure(12 * R);
        for_each_host_chunk(c, host_cols, n_cols, N, [&](uint32_t c0, uint32_t nc, bool first) {
            const uint32_t width = std::min(round_up(nc, 8), pitch - c0);
            if (first) { record(c, GL_STAGE_TRANSPOSE); record(c, GL_STAGE_INTT); record(c, GL_STAGE_LDE); }   // h2d = first chunk
            lde_columns(c, c->in_stage.p + (uint64_t)c0 * N, N, c0, nc, width, log_n, rate_bits, is_coeffs, c->vals.p, t->coeffs.p, pitch,
                        t->leaves.p, pitch, 8, false);
            if (hash_per_chunk) {
                const bool last = c0 + nc == n_cols;
                leaf_absorb(c, t->leaves.p, R, n_cols, pitch, cap_height, c0, c0 + nc, c->hash_state.p, t->digests.p, t->d_cap.p, c0 == 0, last,
                            &c->launches[GL_STAGE_LEAF_HASH]);
                leaves_hashed = leaves_hashed || last;
            }
        }, hash_per_chunk);
    } else {
        record(c, GL_STAGE_TRANSPOSE);
        lde_stage(c, d_cols_in, col_stride, n_cols, log_n, rate_bits, is_coeffs, t->coeffs.p, pitch, t->leaves.p, pitch);
    }
    // Copy-back of the coefficients and the leaves (a host that materialises PolynomialBatch::polynomials / MerkleTree::leaves) leaves
    // on the copy stream as soon as the LDE is done, i.e. PCIe runs while the tree is hashed; only the digests wait for the hash.
    const bool early_copyback = out_coeffs || out_leaves;
    if (out_coeffs) {
        // row-major [N][pitch] -> column-major [n_cols][N] on the device, then one contiguous copy
        c->scratch.ensure(N * n_cols);
        dim3 tb(32, 8), tg((uint32_t)((N + 31) / 32), (n_cols + 31) / 32);
        ntt::transpose_out_kernel<<<tg, tb, 0, c->stream>>>(t->coeffs.p, pitch, c->scratch.p, N, n_cols, N);
        CUDA_CHECK(cudaGetLastError());
        c->launches[GL_STAGE_D2H]++;
    }
    record(c, GL_STAGE_LEAF_HASH);
    if (early_copyback) CUDA_CHECK(cudaEventRecord(c->ev_sync, c->stream));
    if (leaves_hashed) {
        CUDA_CHECK(cudaEventRecord(c->ev[GL_STAGE_TREE], c->stream));
        merkle_levels(c, R, cap_height, t->digests.p, t->d_cap.p, &c->launches[GL_STAGE_TREE]);
    } else {
        merkle_build(c, t->leaves.p, R, n_cols, pitch, cap_height, t->digests.p, t->d_cap.p, &c->launches[GL_STAGE_LEAF_HASH],
                     &c->launches[GL_STAGE_TREE], c->ev[GL_STAGE_TREE]);
    }
    record(c, GL_STAGE_D2H);
    if (early_copyback) {
        // enqueued after the hash kernels were launched: with pageable host memory these calls block the host thread while they
        // run, and the GPU is already hashing by then — the overlap holds for a plain Vec / numpy array as well as for pinned memory
        CUDA_CHECK(cudaStreamWaitEvent(c->copy_stream, c->ev_sync, 0));
        if (out_coeffs) CUDA_CHECK(cudaMemcpyAsync(out_coeffs, c->scratch.p, N * n_cols * 8, cudaMemcpyDeviceToHost, c->copy_stream));
        if (out_leaves)
            CUDA_CHECK(cudaMemcpy2DAsync(out_leaves, (size_t)n_cols * 8, t->leaves.p, (size_t)pitch * 8, (size_t)n_cols * 8, R,
                                         cudaMemcpyDeviceToHost, c->copy_stream));
        CUDA_CHECK(cudaEventRecord(c->ev_copyback, c->copy_stream));
    }
    CUDA_CHECK(cudaMemcpyAsync(t->cap.data(), t->d_cap.p, (32ULL << cap_height), cudaMemcpyDeviceToHost, c->stream));
    if (out_digests && t->n_digests())
        CUDA_CHECK(cudaMemcpyAsync(out_digests, t->digests.p, t->n_digests() * 32, cudaMemcpyDeviceToHost, c->stream));
    if (early_copyback) CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->ev_copyback, 0));   // the d2h stage ends when everything has landed
    record(c, GL_N_STAGES);
    read_stages(c, 0, GL_N_STAGES);
    memcpy(out_cap, t->cap.data(), 32ULL << cap_height);
    if (out_batch) *out_batch = c->trees.put(c, std::move(t));
    return GL_OK;
}

// why the last failed call on `c` failed, for gl_ctx_last_error
int set_error(gl_ctx* c, int code, const std::string& msg) {
    c->err = msg;
    return code;
}

// Turns the exception being handled into the return code of a call on `c`.  Call it only from a catch block, with c->mu held.
int fail(gl_ctx* c) {
    try {
        throw;
    } catch (const GlError& e) {
        cudaGetLastError();
        // host buffers are only borrowed: nothing may read or write them after the call returns
        for (cudaStream_t s : {c->stream, c->copy_stream, c->send_stream, c->pull_stream})
            if (s) cudaStreamSynchronize(s);
        return set_error(c, e.code, e.msg);
    } catch (const std::bad_alloc&) {
        return set_error(c, GL_ERR_OOM, "host allocation failed");
    } catch (...) {
        return set_error(c, GL_ERR_CUDA, "unknown error");
    }
}

}  // namespace

// ============================================================================================ extern "C"
#define GL_API_BEGIN(ctx)                        \
    if (!(ctx)) return GL_ERR_INVALID;           \
    std::lock_guard<std::mutex> _lk((ctx)->mu);  \
    try {                                        \
        CUDA_CHECK(cudaSetDevice((ctx)->device));
#define GL_API_END(ctx)                          \
    }                                            \
    catch (...) {                                \
        return fail(ctx);                        \
    }

extern "C" {

int gl_abi_version(void) { return GL_ABI_VERSION; }

int gl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* gl_strerror(int code) {
    switch (code) {
        case GL_OK: return "ok";
        case GL_ERR_INVALID: return "invalid argument";
        case GL_ERR_CUDA: return "CUDA error";
        case GL_ERR_OOM: return "out of memory";
        case GL_ERR_HANDLE: return "unknown handle";
        case GL_ERR_UNSUPPORTED: return "unsupported shape";
        default: return "unknown error code";
    }
}

int gl_ctx_create(gl_ctx** out, int device) {
    if (!out) return GL_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return GL_ERR_CUDA; }
    if (device < 0 || device >= n) return GL_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return GL_ERR_CUDA;
    gl_ctx* c = new (std::nothrow) gl_ctx;
    if (!c) return GL_ERR_OOM;
    c->device = device;
    auto cuda_failed = [c] { delete c; return GL_ERR_CUDA; };
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) return cuda_failed();
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return cuda_failed();
    {
        int lo = 0, hi = 0;   // the streamed coset plan's few iNTT CTAs must get SM slots as hashing CTAs retire, not queue behind a whole grid
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&c->send_stream, cudaStreamNonBlocking, hi) != cudaSuccess) return cuda_failed();
    }
    for (int i = 0; i < 2; i++)
        if (cudaEventCreateWithFlags(&c->ev_ntt[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_sent[i], cudaEventDisableTiming) != cudaSuccess) return cuda_failed();
    if (cudaStreamCreateWithFlags(&c->pull_stream, cudaStreamNonBlocking) != cudaSuccess) return cuda_failed();
    if (const char* m = getenv("GL_TRACE")) c->trace = atoi(m) != 0;
    if (cudaEventCreateWithFlags(&c->ev_sync, cudaEventDisableTiming) != cudaSuccess) return cuda_failed();
    if (cudaEventCreateWithFlags(&c->ev_copyback, cudaEventDisableTiming) != cudaSuccess) return cuda_failed();
    for (auto& e : c->ev)
        if (cudaEventCreate(&e) != cudaSuccess) return cuda_failed();
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    *out = c;
    return GL_OK;
}

void gl_ctx_destroy(gl_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    c->trees.live.clear();
    c->fris.live.clear();
    c->openings.live.clear();
    c->quotients.live.clear();
    c->roots.clear();
    c->pass_roots.clear();
    c->lde_tables.clear();
    c->coset_cache.clear();
    c->in_stage.release(); c->vals.release(); c->scratch.release(); c->hash_state.release(); c->sync_err.release();
    DevPool::get().trim(c->device);
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->chunk_ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->pull_ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->own_ev) if (e) cudaEventDestroy(e);
    if (c->ev_sync) cudaEventDestroy(c->ev_sync);
    if (c->ev_copyback) cudaEventDestroy(c->ev_copyback);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    if (c->send_stream) { cudaStreamSynchronize(c->send_stream); cudaStreamDestroy(c->send_stream); }
    if (c->pull_stream) { cudaStreamSynchronize(c->pull_stream); cudaStreamDestroy(c->pull_stream); }
    for (int i = 0; i < 2; i++) { if (c->ev_ntt[i]) cudaEventDestroy(c->ev_ntt[i]); if (c->ev_sent[i]) cudaEventDestroy(c->ev_sent[i]); }
    c->send_buf[0].release(); c->send_buf[1].release();
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* gl_ctx_last_error(gl_ctx* c) {
    // the message is copied under the context's mutex into a buffer owned by the CALLING thread: a second thread that shares the
    // context and fails concurrently can no longer invalidate the pointer the first one is reading (valid until this thread's next call)
    if (!c) return "null context";
    static thread_local std::string tls_err;
    std::lock_guard<std::mutex> lk(c->mu);
    tls_err = c->err;
    return tls_err.c_str();
}
uint64_t gl_ctx_stream(gl_ctx* c) { return c ? (uint64_t)(uintptr_t)c->stream : 0; }

int gl_commit(gl_ctx* c, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height,
              int input_is_coeffs, uint64_t* out_coeffs, uint64_t* out_leaves, uint64_t* out_digests, uint64_t* out_cap,
              gl_handle* out_batch) {
    GL_API_BEGIN(c)
    if (!cols) GL_THROW(GL_ERR_INVALID, "cols is NULL");
    return commit_impl(c, cols, nullptr, 0, n_cols, log_n, rate_bits, cap_height, input_is_coeffs, out_coeffs, out_leaves,
                       out_digests, out_cap, out_batch);
    GL_API_END(c)
}

int gl_dev_commit(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
                  uint32_t cap_height, int input_is_coeffs, uint64_t* out_cap, gl_handle* out_batch) {
    GL_API_BEGIN(c)
    if (!d_cols) GL_THROW(GL_ERR_INVALID, "d_cols is NULL");
    return commit_impl(c, nullptr, d_cols, col_stride, n_cols, log_n, rate_bits, cap_height, input_is_coeffs, nullptr, nullptr,
                       nullptr, out_cap, out_batch);
    GL_API_END(c)
}

int gl_dev_lde(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
               int input_is_coeffs, uint64_t* d_out_rows, uint32_t out_pitch, uint64_t* d_out_coeffs) {
    GL_API_BEGIN(c)
    check_shape(n_cols, log_n, rate_bits, 0);
    if (!d_cols || !d_out_rows) GL_THROW(GL_ERR_INVALID, "NULL device pointer");
    if (out_pitch % 4 || out_pitch < n_cols) GL_THROW(GL_ERR_INVALID, "out_pitch must be a multiple of 4 and >= n_cols");
    uint64_t* coeffs = d_out_coeffs;
    if (!coeffs) { c->scratch.ensure(((uint64_t)1 << log_n) * out_pitch); coeffs = c->scratch.p; }
    get_roots(c, log_n);
    get_lde_tables(c, log_n, rate_bits);
    reset_stages(c, GL_STAGE_H2D, GL_STAGE_LEAF_HASH);
    record(c, GL_STAGE_TRANSPOSE);
    lde_stage(c, d_cols, col_stride, n_cols, log_n, rate_bits, input_is_coeffs, coeffs, out_pitch, d_out_rows, out_pitch);
    record(c, GL_STAGE_LEAF_HASH);
    read_stages(c, GL_STAGE_TRANSPOSE, GL_STAGE_LEAF_HASH);
    return GL_OK;
    GL_API_END(c)
}

static int lde_scatter_impl(gl_ctx* c, const uint64_t* d_cols, const uint64_t* const* host_cols, uint64_t col_stride, uint32_t n_cols,
                            uint32_t log_n, uint32_t rate_bits, int input_is_coeffs, uint64_t* const* peer_leaves, uint32_t n_peers,
                            uint32_t leaf_pitch, uint32_t col_off, uint64_t* d_out_coeffs, uint32_t coeff_pitch, uint32_t first_coset,
                            int self_hint = -1) {
    check_shape(n_cols, log_n, rate_bits, 0);
    if ((!d_cols && !host_cols) || !peer_leaves || !d_out_coeffs) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_peers == 0 || (n_peers & (n_peers - 1)) || n_peers > ntt::MAX_PEERS) GL_THROW(GL_ERR_INVALID, "n_peers must be a power of two <= %d", ntt::MAX_PEERS);
    const uint64_t N = 1ULL << log_n, R = N << rate_bits;
    if (R < n_peers) GL_THROW(GL_ERR_INVALID, "fewer leaf rows than peers");
    const int G = column_group(n_cols, coeff_pitch);
    if (col_off + n_cols > leaf_pitch) GL_THROW(GL_ERR_INVALID, "columns do not fit the leaf pitch");
    ntt::Scatter sc{};
    for (uint32_t q = 0; q < n_peers; q++) {
        if (!peer_leaves[q]) GL_THROW(GL_ERR_INVALID, "peer_leaves[%u] is NULL", q);
        sc.peer[q] = peer_leaves[q];
    }
    sc.log_rows_per_peer = log2_exact(R / n_peers);
    sc.col0 = col_off;
    sc.pitch = leaf_pitch;
    sc.ncols = n_cols;
    sc.self = ntt::MAX_PEERS;                 // which peer buffer is this rank's own (allocated by gl_dev_ipc_alloc on this context)?
    for (uint32_t q = 0; q < n_peers; q++)
        if (c->own_ipc.count(peer_leaves[q])) { sc.self = q; break; }
    if (self_hint >= 0 && (uint32_t)self_hint < n_peers) sc.self = (uint32_t)self_hint;   // gl_commit_multi knows its rank
    get_roots(c, log_n);
    get_lde_tables(c, log_n, rate_bits);
    c->scratch.ensure(N * coeff_pitch);      // pass scratch of one coset
    if (!input_is_coeffs) c->vals.ensure(N * coeff_pitch);
    c->send_buf[0].ensure(N * coeff_pitch);
    c->send_buf[1].ensure(N * coeff_pitch);
    reset_stages(c, GL_STAGE_H2D, GL_STAGE_LEAF_HASH);
    if (host_cols) {
        record(c, GL_STAGE_H2D);
        for_each_host_chunk(c, host_cols, n_cols, N, [&](uint32_t c0, uint32_t nc, bool first) {
            const uint32_t width = std::min(round_up(nc, (uint32_t)G), coeff_pitch - c0);
            if (first) { record(c, GL_STAGE_TRANSPOSE); record(c, GL_STAGE_INTT); record(c, GL_STAGE_LDE); }
            lde_columns(c, c->in_stage.p + (uint64_t)c0 * N, N, c0, nc, width, log_n, rate_bits, input_is_coeffs, c->vals.p, d_out_coeffs,
                        coeff_pitch, c->scratch.p, coeff_pitch, G, false, &sc, first_coset);
        });
    } else {
        record(c, GL_STAGE_TRANSPOSE);
        lde_columns(c, d_cols, col_stride, 0, n_cols, coeff_pitch, log_n, rate_bits, input_is_coeffs, c->vals.p, d_out_coeffs, coeff_pitch,
                    c->scratch.p, coeff_pitch, G, true, &sc, first_coset);
    }
    for (int b = 0; b < 2; b++)              // join the shipments: the LDE stage ends when the last coset has left
        if (c->sent_pending[b]) { CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->ev_sent[b], 0)); c->sent_pending[b] = false; }
    record(c, GL_STAGE_LEAF_HASH);
    read_stages(c, host_cols ? GL_STAGE_H2D : GL_STAGE_TRANSPOSE, GL_STAGE_LEAF_HASH);
    if (c->trace && c->trace_ev.size() > 1) {
        cudaStreamSynchronize(c->send_stream);
        fprintf(stderr, "[gl trace dev %d] coset: ntt start-end | send start-end (ms)\n", c->device);
        for (size_t i = 1; i + 3 < c->trace_ev.size(); i += 4) {
            float t[4];
            for (int j = 0; j < 4; j++) cudaEventElapsedTime(&t[j], c->trace_ev[0], c->trace_ev[i + j]);
            fprintf(stderr, "[gl trace dev %d] %2zu: %7.3f-%7.3f | %7.3f-%7.3f\n", c->device, (i - 1) / 4, t[0], t[1], t[2], t[3]);
        }
        for (auto e : c->trace_ev) cudaEventDestroy(e);
        c->trace_ev.clear();
    }
    return GL_OK;
}

int gl_dev_lde_scatter(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
                       int input_is_coeffs, uint64_t* const* peer_leaves, uint32_t n_peers, uint32_t leaf_pitch, uint32_t col_off,
                       uint64_t* d_out_coeffs, uint32_t coeff_pitch, uint32_t first_coset) {
    GL_API_BEGIN(c)
    if (!d_cols) GL_THROW(GL_ERR_INVALID, "d_cols is NULL");
    return lde_scatter_impl(c, d_cols, nullptr, col_stride, n_cols, log_n, rate_bits, input_is_coeffs, peer_leaves, n_peers, leaf_pitch,
                            col_off, d_out_coeffs, coeff_pitch, first_coset);
    GL_API_END(c)
}

int gl_lde_scatter(gl_ctx* c, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits, int input_is_coeffs,
                   uint64_t* const* peer_leaves, uint32_t n_peers, uint32_t leaf_pitch, uint32_t col_off, uint64_t* d_out_coeffs,
                   uint32_t coeff_pitch, uint32_t first_coset) {
    GL_API_BEGIN(c)
    if (!cols) GL_THROW(GL_ERR_INVALID, "cols is NULL");
    return lde_scatter_impl(c, nullptr, cols, 0, n_cols, log_n, rate_bits, input_is_coeffs, peer_leaves, n_peers, leaf_pitch, col_off,
                            d_out_coeffs, coeff_pitch, first_coset);
    GL_API_END(c)
}

// ---- coset-sharded commit: exchange coefficients, evaluate only the cosets this rank owns (include/gl_commit.h) ---------------------
// iNTT of a column shard from device (d_cols) or host columns into the row-major [N][coeff_pitch] coefficients the peers pull
static int intt_impl(gl_ctx* c, const uint64_t* d_cols, const uint64_t* const* host_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n,
                     int input_is_coeffs, uint64_t* d_out_coeffs, uint32_t coeff_pitch) {
    check_shape(n_cols, log_n, 0, 0);
    const int G = column_group(n_cols, coeff_pitch);
    const uint64_t N = 1ULL << log_n;
    get_roots(c, log_n);
    if (!input_is_coeffs) c->vals.ensure(N * coeff_pitch);
    reset_stages(c, GL_STAGE_H2D, GL_STAGE_LEAF_HASH);
    if (host_cols) {
        record(c, GL_STAGE_H2D);
        // the shard crosses PCIe in chunks; transpose + iNTT of chunk k run while chunk k+1 is on the wire
        for_each_host_chunk(c, host_cols, n_cols, N, [&](uint32_t c0, uint32_t nc, bool first) {
            const uint32_t width = std::min(round_up(nc, (uint32_t)G), coeff_pitch - c0);
            if (first) { record(c, GL_STAGE_TRANSPOSE); record(c, GL_STAGE_INTT); }
            intt_columns(c, c->in_stage.p + (uint64_t)c0 * N, N, nc, width, log_n, input_is_coeffs ? nullptr : c->vals.p + c0, d_out_coeffs + c0,
                         coeff_pitch, G, false);
        });
        record(c, GL_STAGE_LDE);
    } else {
        record(c, GL_STAGE_TRANSPOSE);
        intt_columns(c, d_cols, col_stride, n_cols, coeff_pitch, log_n, input_is_coeffs ? nullptr : c->vals.p, d_out_coeffs, coeff_pitch, G, true);
    }
    read_stages(c, host_cols ? GL_STAGE_H2D : GL_STAGE_TRANSPOSE, GL_STAGE_LDE);
    return GL_OK;
}

int gl_dev_intt(gl_ctx* c, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, int input_is_coeffs,
                uint64_t* d_out_coeffs, uint32_t coeff_pitch) {
    GL_API_BEGIN(c)
    if (!d_cols || !d_out_coeffs) GL_THROW(GL_ERR_INVALID, "NULL device pointer");
    return intt_impl(c, d_cols, nullptr, col_stride, n_cols, log_n, input_is_coeffs, d_out_coeffs, coeff_pitch);
    GL_API_END(c)
}

int gl_intt_host(gl_ctx* c, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, int input_is_coeffs, uint64_t* d_out_coeffs,
                 uint32_t coeff_pitch) {
    GL_API_BEGIN(c)
    if (!cols || !d_out_coeffs) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    return intt_impl(c, nullptr, cols, 0, n_cols, log_n, input_is_coeffs, d_out_coeffs, coeff_pitch);
    GL_API_END(c)
}

int gl_dev_lde_own_cosets(gl_ctx* c, uint64_t* const* peer_coeffs, uint64_t* const* d_stage, const uint32_t* pitches, const uint32_t* col_counts,
                          const uint32_t* col_offsets, uint32_t n_peers, uint32_t self, uint32_t log_n, uint32_t rate_bits, uint64_t* d_leaves,
                          uint32_t leaf_pitch) {
    GL_API_BEGIN(c)
    if (!peer_coeffs || !d_stage || !pitches || !col_counts || !col_offsets || !d_leaves) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_peers == 0 || (n_peers & (n_peers - 1)) || n_peers > (uint32_t)ntt::MAX_PEERS || self >= n_peers) GL_THROW(GL_ERR_INVALID, "bad peer count / rank");
    if (n_peers > (1u << rate_bits)) GL_THROW(GL_ERR_INVALID, "coset sharding needs n_peers <= 2^rate_bits");
    if (log_n + rate_bits > 31) GL_THROW(GL_ERR_UNSUPPORTED, "log_n + rate_bits > 31");
    const uint64_t N = 1ULL << log_n;
    const uint32_t blocks_per_rank = (1u << rate_bits) / n_peers, first_block = self * blocks_per_rank;
    for (uint32_t q = 0; q < n_peers; q++) {
        if (!peer_coeffs[q] || (q != self && !d_stage[q])) GL_THROW(GL_ERR_INVALID, "peer %u: NULL buffer", q);
        if (pitches[q] % 4 || pitches[q] < col_counts[q] || col_offsets[q] % 4 || col_offsets[q] + col_counts[q] > leaf_pitch)
            GL_THROW(GL_ERR_INVALID, "peer %u: bad column layout", q);
    }
    get_roots(c, log_n);
    const auto& tabs = get_lde_tables(c, log_n, rate_bits);
    ensure_events(c->pull_ev, n_peers);
    reset_stages(c, GL_STAGE_LDE, GL_STAGE_LEAF_HASH);
    record(c, GL_STAGE_LDE);
    // every pull is enqueued up front on the copy stream, nearest neighbour first (rank q pulls from q+1, q+2, ...: at any moment every
    // rank reads from a different peer); the compute stream takes the blocks in the same order, own block first
    CUDA_CHECK(cudaEventRecord(c->ev_sync, c->stream));
    CUDA_CHECK(cudaStreamWaitEvent(c->pull_stream, c->ev_sync, 0));        // staging buffers may still be read by an earlier call's NTTs
    cudaEvent_t tr0 = nullptr, tr1 = nullptr;
    uint64_t pulled_bytes = 0;
    if (c->trace) { cudaEventCreate(&tr0); cudaEventCreate(&tr1); cudaEventRecord(tr0, c->pull_stream); }
    for (uint32_t k = 1; k < n_peers; k++) pulled_bytes += N * pitches[(self + k) % n_peers] * 8;
    for (uint32_t k = 1; k < n_peers; k++) {
        const uint32_t q = (self + k) % n_peers;
        CUDA_CHECK(cudaMemcpyAsync(d_stage[q], peer_coeffs[q], N * pitches[q] * 8, cudaMemcpyDefault, c->pull_stream));
        CUDA_CHECK(cudaEventRecord(c->pull_ev[q], c->pull_stream));
    }
    if (c->trace) cudaEventRecord(tr1, c->pull_stream);
    for (uint32_t k = 0; k < n_peers; k++) {
        const uint32_t q = (self + k) % n_peers;
        const uint64_t* coeffs = q == self ? peer_coeffs[q] : d_stage[q];
        if (q != self) CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->pull_ev[q], 0));
        const int G = (column_group(col_counts[q], pitches[q]) == 4 || pitches[q] % 8) ? 4 : 8;   // 8-column tiles need a pitch of whole groups
        for (uint32_t b = 0; b < blocks_per_rank; b++) {
            const uint32_t s = h_bitrev(first_block + b, rate_bits);       // leaf block b of the batch is LDE coset bitrev_r(b)
            uint64_t* dst = d_leaves + (uint64_t)b * N * leaf_pitch + col_offsets[q];
            run_ntt(c, const_cast<uint64_t*>(coeffs), pitches[q], dst, leaf_pitch, round_up(col_counts[q], (uint32_t)G), log_n, false, &tabs[s], G,
                    &c->launches[GL_STAGE_LDE]);
        }
    }
    record(c, GL_STAGE_LEAF_HASH);
    read_stages(c, GL_STAGE_LDE, GL_STAGE_LEAF_HASH);
    if (c->trace) {   // NVLink ingress of this rank: the G-1 coefficient blocks, back to back on the copy engine
        cudaStreamSynchronize(c->pull_stream);
        float ms = 0;
        cudaEventElapsedTime(&ms, tr0, tr1);
        fprintf(stderr, "[gl trace dev %d] coset plan: pulled %.1f MB from %u peers in %.3f ms = %.1f GB/s (NVLink ingress); LDE stage %.3f ms\n", c->device,
                pulled_bytes / 1e6, n_peers - 1, ms, ms > 0 ? pulled_bytes / ms / 1e6 : 0.0, c->stage_ms[GL_STAGE_LDE]);
        cudaEventDestroy(tr0); cudaEventDestroy(tr1);
    }
    return GL_OK;
    GL_API_END(c)
}

// ---- coset-sharded commit streamed from host columns (include/gl_commit.h · gl_commit_coset_stream) ---------------------------------
namespace {
struct StreamLayout {
    uint32_t G, gw, n_groups, W, C;
    bool has(uint32_t q, uint32_t w) const { return w * G + q < n_groups; }
    uint32_t cols(uint32_t q, uint32_t w) const { return has(q, w) ? std::min(gw, C - gw * (w * G + q)) : 0; }
    uint32_t own_cols(uint32_t q) const { uint32_t n = 0; for (uint32_t w = 0; w < W; w++) n += cols(q, w); return n; }
};
StreamLayout stream_layout(const gl_stream_plan_t* p) {
    if (!p) GL_THROW(GL_ERR_INVALID, "plan is NULL");
    if (p->group_width != 4 && p->group_width != 8) GL_THROW(GL_ERR_INVALID, "group_width must be 4 or 8");
    if (p->n_peers == 0 || (p->n_peers & (p->n_peers - 1)) || p->n_peers > (uint32_t)ntt::MAX_PEERS || p->self >= p->n_peers)
        GL_THROW(GL_ERR_INVALID, "bad peer count / rank");
    if (p->n_peers > (1u << p->rate_bits)) GL_THROW(GL_ERR_INVALID, "coset sharding needs n_peers <= 2^rate_bits");
    if ((p->n_peers * p->group_width) % 8) GL_THROW(GL_ERR_INVALID, "a wave (n_peers * group_width columns) must be a multiple of the sponge rate 8");
    if (p->n_cols <= 4) GL_THROW(GL_ERR_UNSUPPORTED, "leaves of <= 4 elements are not hashed (hash_or_noop): use gl_dev_merkle");
    if (p->log_n + p->rate_bits > 31) GL_THROW(GL_ERR_UNSUPPORTED, "log_n + rate_bits > 31");
    if (p->leaf_pitch % 8 || p->leaf_pitch < round_up(p->n_cols, 8u)) GL_THROW(GL_ERR_INVALID, "leaf_pitch must be a multiple of 8 and >= round_up(n_cols, 8)");
    const uint32_t log_rows = p->log_n + p->rate_bits - log2_exact(p->n_peers);
    if (p->cap_height > log_rows) GL_THROW(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len()) of the rank's leaf range");
    StreamLayout L;
    L.G = p->n_peers; L.gw = p->group_width; L.C = p->n_cols;
    L.n_groups = (p->n_cols + L.gw - 1) / L.gw;
    L.W = (L.n_groups + L.G - 1) / L.G;
    return L;
}
}  // namespace

int gl_stream_plan_sizes(const gl_stream_plan_t* plan, uint64_t* exported_words, uint64_t* stage_words, uint32_t* n_waves, uint32_t* n_own_cols) {
    try {
        const StreamLayout L = stream_layout(plan);
        const uint64_t N = 1ULL << plan->log_n;
        if (exported_words) *exported_words = (uint64_t)L.W * N * L.gw + (uint64_t)L.G * L.W;
        if (stage_words) *stage_words = (uint64_t)L.G * L.W * N * L.gw;
        if (n_waves) *n_waves = L.W;
        if (n_own_cols) *n_own_cols = L.own_cols(plan->self);
        return GL_OK;
    } catch (const GlError& e) {
        return e.code;
    }
}

namespace {
// d_cap: device buffer for the rank's subtree roots (nullptr: the context's scratch)
void coset_stream_impl(gl_ctx* c, const gl_stream_plan_t* plan, const uint64_t* const* own_cols, int input_is_coeffs, uint64_t* const* peer_bufs,
                       uint64_t* d_stage, uint64_t* d_leaves, uint64_t* d_digests, uint64_t* d_cap, uint64_t* out_cap) {
    const StreamLayout L = stream_layout(plan);
    if (!peer_bufs || !d_stage || !d_leaves || !d_digests || !out_cap) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    const uint32_t G = L.G, gw = L.gw, W = L.W, self = plan->self, log_n = plan->log_n, rate_bits = plan->rate_bits, C = L.C;
    const uint32_t n_own = L.own_cols(self);
    if (n_own && !own_cols) GL_THROW(GL_ERR_INVALID, "own_cols is NULL");
    for (uint32_t j = 0; j < n_own; j++)
        if (!own_cols[j]) GL_THROW(GL_ERR_INVALID, "own_cols[%u] is NULL", j);
    for (uint32_t q = 0; q < G; q++)
        if (!peer_bufs[q]) GL_THROW(GL_ERR_INVALID, "peer %u: NULL buffer", q);
    const uint64_t N = 1ULL << log_n, blk = N * gw;                     // words of one (rank, wave) coefficient block [N][gw]
    const uint32_t blocks_per_rank = (1u << rate_bits) / G, first_block = self * blocks_per_rank;
    const uint64_t rows = (uint64_t)blocks_per_rank * N;
    const uint32_t cap_height = plan->cap_height, leaf_pitch = plan->leaf_pitch;
    const uint64_t flags_off = (uint64_t)W * blk;
    uint64_t* own_buf = peer_bufs[self];
    preload_stream_kernels();
    get_roots(c, log_n);
    const auto& tabs = get_lde_tables(c, log_n, rate_bits);
    for (uint32_t a : plan_passes(log_n, 10)) get_pass_roots(c, a);      // (created with a stream synchronise: not while a wait is parked)
    c->in_stage.ensure(blk * W);
    if (!input_is_coeffs) c->vals.ensure(blk * W);
    c->hash_state.ensure(12 * rows);
    c->sync_err.ensure(1);
    if (!d_cap) {
        c->scratch.ensure(std::max<uint64_t>(4ULL << cap_height, 1));
        d_cap = c->scratch.p;
    }
    ensure_events(c->chunk_ev, W);
    ensure_events(c->own_ev, W);
    ensure_events(c->pull_ev, (size_t)W * G);
    uint64_t timeout_ns = 20000ULL * 1000000ULL;
    if (const char* m = getenv("GL_PEER_TIMEOUT_MS")) timeout_ns = strtoull(m, nullptr, 10) * 1000000ULL;
    const uint64_t ticket0 = plan->epoch * W + 1;                        // wave w publishes ticket0 + w
    reset_stages(c, 0, GL_N_STAGES);

    record(c, GL_STAGE_H2D);
    CUDA_CHECK(cudaMemsetAsync(c->sync_err.p, 0, 8, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev_sync, c->stream));                  // staging / in_stage may still be read by an earlier call
    for (cudaStream_t st : {c->copy_stream, c->send_stream, c->pull_stream}) CUDA_CHECK(cudaStreamWaitEvent(st, c->ev_sync, 0));

    // (1) copy stream: the own group of every wave, host -> device
    for (uint32_t w = 0, j = 0; w < W; w++) {
        for (uint32_t k = 0; k < L.cols(self, w); k++, j++)
            CUDA_CHECK(cudaMemcpyAsync(c->in_stage.p + w * blk + (uint64_t)k * N, own_cols[j], N * 8, cudaMemcpyHostToDevice, c->copy_stream));
        CUDA_CHECK(cudaEventRecord(c->chunk_ev[w], c->copy_stream));
    }
    // (2) high-priority stream: transpose + iNTT of the own group into the exported block, then the ticket to every peer.  These few CTAs
    //     take SM slots as hashing CTAs retire, so a group is published as soon as it has landed, whatever the compute stream is doing.
    {
        struct UseStream {
            gl_ctx* c; cudaStream_t saved;
            UseStream(gl_ctx* c, cudaStream_t s) : c(c), saved(c->stream) { c->stream = s; }
            ~UseStream() { c->stream = saved; }
        } on_prep(c, c->send_stream);
        for (uint32_t w = 0; w < W; w++) {
            const uint32_t nc = L.cols(self, w);
            if (!nc) continue;
            CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->chunk_ev[w], 0));
            intt_columns(c, c->in_stage.p + w * blk, N, nc, gw, log_n, input_is_coeffs ? nullptr : c->vals.p + w * blk, own_buf + w * blk, gw,
                         (int)gw, false);
            CUDA_CHECK(cudaEventRecord(c->own_ev[w], c->stream));
            if (G > 1) {
                peersync::Slots s{};
                for (uint32_t q = 0; q < G; q++) s.p[q] = q == self ? nullptr : peer_bufs[q] + flags_off + (uint64_t)self * W + w;
                peersync::signal_kernel<<<1, 32, 0, c->stream>>>(s, G, ticket0 + w);
                CUDA_CHECK(cudaGetLastError());
            }
        }
    }
    // (3) pull stream: wait for the peer's ticket in the OWN flag array, then one contiguous copy-engine pull per (wave, peer), nearest
    //     neighbour first (at any moment every rank reads from a different peer)
    for (uint32_t w = 0; w < W; w++)
        for (uint32_t k = 1; k < G; k++) {
            const uint32_t q = (self + k) % G;
            if (!L.has(q, w)) continue;
            peersync::wait_kernel<<<1, 1, 0, c->pull_stream>>>(own_buf + flags_off + (uint64_t)q * W + w, ticket0 + w, reinterpret_cast<uint32_t*>(c->sync_err.p),
                                                              timeout_ns);
            CUDA_CHECK(cudaGetLastError());
            CUDA_CHECK(cudaMemcpyAsync(d_stage + ((uint64_t)q * W + w) * blk, peer_bufs[q] + w * blk, blk * 8, cudaMemcpyDefault, c->pull_stream));
            CUDA_CHECK(cudaEventRecord(c->pull_ev[(size_t)w * G + q], c->pull_stream));
        }
    // (4) compute stream: own cosets of the wave's groups as they arrive (own group first), then the wave's columns into the leaf sponge
    bool started = false;
    std::vector<cudaEvent_t> tr;                                          // GL_TRACE=1: per wave {first group ready, NTTs done, absorbed}
    auto mark = [&]() {
        if (!c->trace) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->stream); tr.push_back(e);
    };
    // One launch per pass covers all groups of the wave: the first pass reads every group from the block it arrived in (run_ntt's
    // src_list), the later passes run in place on the wave's adjacent leaf columns with 8-column tiles.  (Per-group launches — 4-column
    // transforms of 32-byte row segments, 16 small launches per wave at 8 GPUs — measured 0.95 ms per wave against 0.6 for this form.)
    // The FIRST wave keeps per-group launches: its groups arrive one by one behind the slowest rank's copy, and transforming each as it
    // lands hides the NTTs behind the remaining pulls (8 GPUs: first wave done at 3.3 ms instead of 3.9).
    const bool can_merge = log_n >= 3;
    for (uint32_t w = 0; w < W; w++) {
        const bool one_launch = can_merge && w > 0;
        bool first_in_wave = true;
        const uint64_t* srcs[ntt::MAX_PEERS] = {};
        uint32_t n_src = 0;
        for (uint32_t k = 0; k < G; k++) {
            const uint32_t q = (self + k) % G;
            if (!L.has(q, w)) continue;
            CUDA_CHECK(cudaStreamWaitEvent(c->stream, q == self ? c->own_ev[w] : c->pull_ev[(size_t)w * G + q], 0));
            if (first_in_wave) { mark(); first_in_wave = false; }
            if (!started) { record(c, GL_STAGE_TRANSPOSE); record(c, GL_STAGE_INTT); record(c, GL_STAGE_LDE); started = true; }   // h2d = until the first group is ready
            uint64_t* coeffs = q == self ? own_buf + w * blk : d_stage + ((uint64_t)q * W + w) * blk;
            srcs[q] = coeffs;                                            // the groups a wave has are q = 0 .. n_src-1 (a prefix)
            n_src = std::max(n_src, q + 1);
            if (one_launch) continue;
            for (uint32_t b = 0; b < blocks_per_rank; b++) {
                const uint32_t s = h_bitrev(first_block + b, rate_bits);   // leaf block b of the batch is LDE coset bitrev_r(b)
                uint64_t* dst = d_leaves + (uint64_t)b * N * leaf_pitch + (uint64_t)gw * (w * G + q);
                run_ntt(c, coeffs, gw, dst, leaf_pitch, gw, log_n, false, &tabs[s], (int)gw, &c->launches[GL_STAGE_LDE]);
            }
        }
        if (one_launch)
            for (uint32_t b = 0; b < blocks_per_rank; b++) {
                const uint32_t s = h_bitrev(first_block + b, rate_bits);
                uint64_t* dst = d_leaves + (uint64_t)b * N * leaf_pitch + (uint64_t)gw * w * G;
                run_ntt(c, nullptr, gw, dst, leaf_pitch, n_src * gw, log_n, false, &tabs[s], (int)gw, &c->launches[GL_STAGE_LDE], nullptr, srcs);
            }
        mark();
        const uint32_t c0 = w * G * gw, c1 = std::min(C, (w + 1) * G * gw);
        leaf_absorb(c, d_leaves, rows, C, leaf_pitch, cap_height, c0, c1, c->hash_state.p, d_digests, d_cap, w == 0, w + 1 == W, &c->launches[GL_STAGE_LEAF_HASH]);
        mark();
    }
    record(c, GL_STAGE_LEAF_HASH);
    record(c, GL_STAGE_TREE);
    merkle_levels(c, rows, cap_height, d_digests, d_cap, &c->launches[GL_STAGE_TREE]);
    record(c, GL_STAGE_D2H);
    uint64_t err = 0;
    CUDA_CHECK(cudaMemcpyAsync(out_cap, d_cap, 32ULL << cap_height, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(&err, c->sync_err.p, 8, cudaMemcpyDeviceToHost, c->stream));
    record(c, GL_N_STAGES);
    read_stages(c, 0, GL_N_STAGES);
    CUDA_CHECK(cudaStreamSynchronize(c->send_stream));                   // (both idle by dependency; the host buffers are only borrowed)
    CUDA_CHECK(cudaStreamSynchronize(c->pull_stream));
    if (c->trace) {
        std::string line;
        char buf[96];
        for (size_t i = 0; i + 2 < tr.size() + 0 && i / 3 < W; i += 3) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, c->ev[GL_STAGE_H2D], tr[i]); cudaEventElapsedTime(&b, c->ev[GL_STAGE_H2D], tr[i + 1]);
            cudaEventElapsedTime(&d, c->ev[GL_STAGE_H2D], tr[i + 2]);
            snprintf(buf, sizeof buf, " w%zu: ready %.2f ntt %.2f absorbed %.2f;", i / 3, a, b, d);
            line += buf;
        }
        float tot = 0;
        cudaEventElapsedTime(&tot, c->ev[GL_STAGE_H2D], c->ev[GL_N_STAGES]);
        fprintf(stderr, "[gl trace dev %d] streamed coset plan (ms from call start):%s end %.2f\n", c->device, line.c_str(), tot);
        for (auto e : tr) cudaEventDestroy(e);
    }
    if (err) GL_THROW(GL_ERR_CUDA, "a peer did not publish its coefficient group within the time limit (GL_PEER_TIMEOUT_MS)");
}
}  // namespace

int gl_commit_coset_stream(gl_ctx* c, const gl_stream_plan_t* plan, const uint64_t* const* own_cols, int input_is_coeffs,
                           uint64_t* const* peer_bufs, uint64_t* d_stage, uint64_t* d_leaves, uint64_t* d_digests, uint64_t* out_cap) {
    GL_API_BEGIN(c)
    coset_stream_impl(c, plan, own_cols, input_is_coeffs, peer_bufs, d_stage, d_leaves, d_digests, nullptr, out_cap);
    return GL_OK;
    GL_API_END(c)
}

// ---- CUDA IPC: one process per GPU, each exports its leaf buffer and maps its peers' (NVLink peer access) -----------
int gl_dev_ipc_alloc(gl_ctx* c, uint64_t words, uint64_t** out_ptr, uint8_t out_handle[64]) {
    GL_API_BEGIN(c)
    if (!out_ptr || !out_handle || words == 0) GL_THROW(GL_ERR_INVALID, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    uint64_t* p = nullptr;
    CUDA_CHECK(cudaMalloc(&p, words * 8));    // not pooled: an exported allocation must stay a whole cudaMalloc block
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); CUDA_CHECK(e); }
    CUDA_CHECK(cudaMemsetAsync(p, 0, words * 8, c->stream));   // the streamed coset plan keeps its ticket words here: they must start at 0
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    memcpy(out_handle, &h, 64);
    *out_ptr = p;
    c->own_ipc.insert(p);
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_ipc_open(gl_ctx* c, const uint8_t handle[64], uint64_t** out_ptr) {
    GL_API_BEGIN(c)
    if (!handle || !out_ptr) GL_THROW(GL_ERR_INVALID, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void* p = nullptr;
    CUDA_CHECK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *out_ptr = (uint64_t*)p;
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_ipc_close(gl_ctx* c, uint64_t* ptr) {
    GL_API_BEGIN(c)
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    if (ptr) CUDA_CHECK(cudaIpcCloseMemHandle(ptr));
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_ipc_free(gl_ctx* c, uint64_t* ptr) {
    GL_API_BEGIN(c)
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    c->own_ipc.erase(ptr);
    if (ptr) CUDA_CHECK(cudaFree(ptr));
    return GL_OK;
    GL_API_END(c)
}

int gl_dev_alloc(gl_ctx* c, uint64_t words, uint64_t** out_ptr) {
    GL_API_BEGIN(c)
    if (!out_ptr || words == 0) GL_THROW(GL_ERR_INVALID, "bad arguments");
    uint64_t* p = nullptr;
    CUDA_CHECK(cudaMalloc(&p, words * 8));
    *out_ptr = p;
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_free(gl_ctx* c, uint64_t* ptr) {
    GL_API_BEGIN(c)
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    if (ptr) CUDA_CHECK(cudaFree(ptr));
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_upload(gl_ctx* c, const uint64_t* host_src, uint64_t* d_dst, uint64_t words) {
    GL_API_BEGIN(c)
    if ((!host_src || !d_dst) && words) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (words) CUDA_CHECK(cudaMemcpyAsync(d_dst, host_src, words * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}
int gl_dev_download(gl_ctx* c, const uint64_t* d_src, uint64_t* host_dst, uint64_t words) {
    GL_API_BEGIN(c)
    if ((!host_dst || !d_src) && words) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (words) CUDA_CHECK(cudaMemcpyAsync(host_dst, d_src, words * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_dev_repack(gl_ctx* c, const uint64_t* d_src, uint32_t src_pitch, uint32_t src_cols, uint64_t n_rows, uint64_t* d_dst,
                  uint32_t dst_pitch, uint32_t dst_col_off) {
    GL_API_BEGIN(c)
    if (!d_src || !d_dst || dst_col_off + src_cols > dst_pitch || src_cols > src_pitch) GL_THROW(GL_ERR_INVALID, "bad repack arguments");
    uint64_t total = n_rows * src_cols;
    if (total) {
        ntt::repitch_kernel<<<(uint32_t)((total + 255) / 256), 256, 0, c->stream>>>(d_src, src_pitch, d_dst, dst_pitch, dst_col_off,
                                                                                  src_cols, n_rows);
        CUDA_CHECK(cudaGetLastError());
    }
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_dev_merkle(gl_ctx* c, const uint64_t* d_leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t pitch, uint32_t cap_height,
                  uint64_t* d_digests, uint64_t* out_cap) {
    GL_API_BEGIN(c)
    if (!d_leaves || !out_cap) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_leaves == 0 || (n_leaves & (n_leaves - 1))) GL_THROW(GL_ERR_INVALID, "n_leaves must be a power of two");
    if ((1ULL << cap_height) > n_leaves) GL_THROW(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len())");
    if (pitch % 8 || pitch < leaf_len) GL_THROW(GL_ERR_INVALID, "pitch must be a multiple of 8 and >= leaf_len");
    if (!d_digests && n_leaves > (1ULL << cap_height)) GL_THROW(GL_ERR_INVALID, "d_digests is NULL");
    c->scratch.ensure(4ULL << cap_height);
    reset_stages(c, GL_STAGE_LEAF_HASH, GL_N_STAGES);
    record(c, GL_STAGE_LEAF_HASH);
    merkle_build(c, d_leaves, n_leaves, leaf_len, pitch, cap_height, d_digests, c->scratch.p, &c->launches[GL_STAGE_LEAF_HASH],
                 &c->launches[GL_STAGE_TREE], c->ev[GL_STAGE_TREE]);
    record(c, GL_STAGE_D2H);
    CUDA_CHECK(cudaMemcpyAsync(out_cap, c->scratch.p, 32ULL << cap_height, cudaMemcpyDeviceToHost, c->stream));
    read_stages(c, GL_STAGE_LEAF_HASH, GL_STAGE_D2H);
    return GL_OK;
    GL_API_END(c)
}

int gl_merkle_new(gl_ctx* c, const uint64_t* leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t cap_height,
                  uint64_t* out_digests, uint64_t* out_cap, gl_handle* out_tree) {
    GL_API_BEGIN(c)
    if (!leaves || !out_cap) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_leaves == 0 || (n_leaves & (n_leaves - 1))) GL_THROW(GL_ERR_INVALID, "n_leaves must be a power of two");
    if (n_leaves > (1ULL << 31)) GL_THROW(GL_ERR_UNSUPPORTED, "too many leaves");
    if ((1ULL << cap_height) > n_leaves)
        GL_THROW(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len()) (cap_height=%u, leaves=%llu)", cap_height,
                 (unsigned long long)n_leaves);
    const uint32_t pitch = round_up(leaf_len ? leaf_len : 1, 8);
    auto t = std::make_unique<Tree>(n_leaves, leaf_len, pitch, cap_height);
    if (leaf_len) {
        // packed host rows -> staging -> [n_leaves][pitch] with every word canonicalised (inputs may be any 64-bit representative;
        // everything gl_tree_get / open_batch / read hands back is canonical, like every other ingest path)
        const uint64_t total = n_leaves * leaf_len;
        c->in_stage.ensure(total);
        CUDA_CHECK(cudaMemcpyAsync(c->in_stage.p, leaves, total * 8, cudaMemcpyHostToDevice, c->stream));
        if (pitch != leaf_len) CUDA_CHECK(cudaMemsetAsync(t->leaves.p, 0, n_leaves * pitch * 8, c->stream));
        ntt::repitch_kernel<<<(uint32_t)((total + 255) / 256), 256, 0, c->stream>>>(c->in_stage.p, leaf_len, t->leaves.p, pitch, 0, leaf_len, n_leaves);
        CUDA_CHECK(cudaGetLastError());
    }
    merkle_build(c, t->leaves.p, n_leaves, leaf_len, pitch, cap_height, t->digests.p, t->d_cap.p, nullptr, nullptr, nullptr);
    finish_tree(c, std::move(t), out_digests, out_cap, out_tree);
    return GL_OK;
    GL_API_END(c)
}

// ---- one process, several GPUs -------------------------------------------------------------------------------------------------
// CircuitData::prove runs in ONE process; a prover that owns several GPUs of the box calls gl_commit_multi with one context per
// device.  Same plan as the one-process-per-GPU path (plonky2.5_b200/sharded.py, DESIGN.md §6): rank g = ctxs[g] runs the iNTT + LDE
// of its column slice (columns dealt in groups of 4 so that every slice starts sector aligned), every coset's rows reach the rank
// that owns that leaf range (peer copies behind the next coset's NTT; own rows stored by the NTT itself), the ranks meet once, and
// every rank hashes its contiguous leaf range = whole cap subtrees.  One worker thread per context; in a single process peer
// buffers are plain device pointers (unified addressing), so there is no IPC.
namespace {
struct HostBarrier {
    std::mutex mu;
    std::condition_variable cv;
    uint32_t n, waiting = 0, phase = 0;
    explicit HostBarrier(uint32_t n_) : n(n_) {}
    void arrive_and_wait() {
        std::unique_lock<std::mutex> lk(mu);
        const uint32_t ph = phase;
        if (++waiting == n) { waiting = 0; phase++; cv.notify_all(); }
        else cv.wait(lk, [&] { return phase != ph; });
    }
};

struct MultiPlan {   // ShardPlan of plonky2.5_b200/sharded.py
    std::vector<uint32_t> col_counts, col_offsets, pitches;
    MultiPlan(uint32_t n_cols, uint32_t world) : col_counts(world), col_offsets(world), pitches(world) {
        const uint32_t n_groups = (n_cols + 3) / 4;
        if (n_groups >= world) {
            const uint32_t base = n_groups / world, rem = n_groups % world;
            for (uint32_t g = 0; g < world; g++) col_counts[g] = 4 * (base + (g < rem ? 1 : 0));
            col_counts[world - 1] -= 4 * n_groups - n_cols;   // the last group may be partial
        } else {
            const uint32_t base = n_cols / world, rem = n_cols % world;
            for (uint32_t g = 0; g < world; g++) col_counts[g] = base + (g < rem ? 1 : 0);
        }
        uint32_t off = 0;
        for (uint32_t g = 0; g < world; g++) {
            col_offsets[g] = off;
            off += col_counts[g];
            const uint32_t c = col_counts[g];
            pitches[g] = (round_up(c, 8) - c < 4) ? round_up(c, 8) : round_up(c, 4);
        }
    }
};
}  // namespace

int gl_commit_multi(gl_ctx* const* ctxs, uint32_t n_ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
                    uint32_t cap_height, int input_is_coeffs, uint64_t* out_cap, gl_handle* out_trees) {
    if (!ctxs || n_ctx == 0 || !ctxs[0]) return GL_ERR_INVALID;
    gl_ctx* c0 = ctxs[0];
    auto fail0 = [&](int code, const std::string& msg) { std::lock_guard<std::mutex> lk(c0->mu); return set_error(c0, code, msg); };
    if ((n_ctx & (n_ctx - 1)) || n_ctx > (uint32_t)ntt::MAX_PEERS) return fail0(GL_ERR_INVALID, "n_ctx must be a power of two <= 16");
    for (uint32_t g = 0; g < n_ctx; g++) {
        if (!ctxs[g]) return fail0(GL_ERR_INVALID, "NULL context");
        for (uint32_t q = 0; q < g; q++)
            if (ctxs[q] == ctxs[g]) return fail0(GL_ERR_INVALID, "the same context appears twice");
    }
    if (!cols || !out_cap || !out_trees) return fail0(GL_ERR_INVALID, "NULL pointer");
    if (n_cols < n_ctx) return fail0(GL_ERR_INVALID, "fewer columns than contexts");
    if (log_n + rate_bits > 31) return fail0(GL_ERR_UNSUPPORTED, "log_n + rate_bits > 31");
    if (cap_height > log_n + rate_bits) return fail0(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len())");
    if ((1ULL << cap_height) < n_ctx) return fail0(GL_ERR_INVALID, "cap_height too small: every context must own at least one whole cap subtree");
    for (uint32_t j = 0; j < n_cols; j++)
        if (!cols[j]) return fail0(GL_ERR_INVALID, "cols[j] is NULL");

    const uint32_t G = n_ctx, log_g = log2_exact(G), local_cap_height = cap_height - log_g;
    const uint64_t N = 1ULL << log_n, R = N << rate_bits, rows_per_rank = R / G;
    const uint32_t leaf_pitch = round_up(n_cols, 8);
    const MultiPlan plan(n_cols, G);
    // Host columns, as many cosets as contexts or more: the STREAMED coset plan (coset_stream_impl) — per wave every context copies and
    // inverse-transforms its column group, the others pull it behind a ticket, each evaluates its own cosets and absorbs the wave into the
    // leaf sponge; the workers never meet between the first and the last barrier.
    // One context per DEVICE only: a ticket wait parks the items queued behind it, and streams of different contexts on one device can share
    // a hardware queue — the peer's signal could sit behind the very wait it is meant to release.  (With one context per device every
    // device's queues only ever hold that context's own work, enqueued copy -> iNTT + signal -> waits -> compute, so nothing a peer depends on
    // is ever behind a wait.)
    bool distinct_devices = true;
    for (uint32_t g = 0; g < n_ctx; g++)
        for (uint32_t q = 0; q < g; q++) distinct_devices = distinct_devices && ctxs[q]->device != ctxs[g]->device;
    // Measured (host columns, 2^20 x 135): 2 devices 2 350 Melem/s streamed against 2 245 with the shipment plan; 8 devices 6 108 against
    // 6 575 — the streamed plan enqueues ~250 launches / copies / events per context and call, and eight worker threads of ONE process push
    // them through the same driver locks (one process per GPU does not pay that: 7 491).  So it is the plan for two contexts only.
    const bool streamed = G <= (1u << rate_bits) && n_cols > 4 && distinct_devices && n_ctx <= 2;
    gl_stream_plan_t sp{};
    sp.n_cols = n_cols; sp.log_n = log_n; sp.rate_bits = rate_bits; sp.cap_height = local_cap_height; sp.n_peers = G;
    sp.group_width = (n_cols >= 4 * 8 * G || G == 1) ? 8 : 4; sp.leaf_pitch = leaf_pitch; sp.epoch = 0;
    uint64_t exported_words = 0, stage_words = 0;
    uint32_t n_waves = 0;
    if (streamed && gl_stream_plan_sizes(&sp, &exported_words, &stage_words, &n_waves, nullptr) != GL_OK) return fail0(GL_ERR_INVALID, "bad streamed plan");
    std::vector<uint64_t*> peer_bufs(G, nullptr);
    std::vector<uint64_t*> peer_leaves(G, nullptr);
    std::vector<std::unique_ptr<Tree>> trees(G);
    std::vector<int> rcs(G, GL_OK);
    HostBarrier barrier(G);

    auto worker = [&](uint32_t g) {
        gl_ctx* c = ctxs[g];
        std::lock_guard<std::mutex> lk(c->mu);
        // every phase is tried separately: a rank that failed still arrives at the barriers, so nobody waits forever
        auto phase = [&](auto&& body) {
            if (rcs[g] != GL_OK) return;
            try {
                body();
            } catch (...) {
                rcs[g] = fail(c);
            }
        };
        phase([&] {   // A: this rank's leaf range, digests and sub-cap; peers become addressable
            CUDA_CHECK(cudaSetDevice(c->device));
            auto t = std::make_unique<Tree>(rows_per_rank, n_cols, leaf_pitch, local_cap_height);
            if (streamed) {
                preload_stream_kernels();            // before the barrier: no context may load a kernel once any device parks a ticket wait
                get_roots(c, log_n);
                get_lde_tables(c, log_n, rate_bits);
                for (uint32_t a : plan_passes(log_n, 10)) get_pass_roots(c, a);
                // exported buffer: this context's coefficient groups [n_waves][N][gw] + the ticket words, which must read 0 before any peer signals
                t->coeffs.ensure(exported_words);
                CUDA_CHECK(cudaMemsetAsync(t->coeffs.p + (exported_words - (uint64_t)G * n_waves), 0, (uint64_t)G * n_waves * 8, c->stream));
                CUDA_CHECK(cudaStreamSynchronize(c->stream));
                peer_bufs[g] = t->coeffs.p;
            } else {
                t->coeffs.ensure(N * plan.pitches[g]);   // this rank's coefficient slice [N][pitch_g] (not served by gl_tree_read: has_coeffs stays false)
            }
            for (uint32_t q = 0; q < G; q++) {
                if (ctxs[q]->device == c->device) continue;
                int can = 0;
                CUDA_CHECK(cudaDeviceCanAccessPeer(&can, c->device, ctxs[q]->device));
                if (!can) GL_THROW(GL_ERR_UNSUPPORTED, "device %d cannot access device %d", c->device, ctxs[q]->device);
                cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else CUDA_CHECK(e);
            }
            peer_leaves[g] = t->leaves.p;
            trees[g] = std::move(t);
        });
        barrier.arrive_and_wait();               // all leaf buffers exist
        bool all_ok = true;
        for (uint32_t q = 0; q < G; q++) all_ok = all_ok && rcs[q] == GL_OK;
        if (all_ok && streamed)
            phase([&] {   // B+C streamed: waves of copy / iNTT / ticket / pull / own cosets / absorb, then the tree above the digests
                CUDA_CHECK(cudaSetDevice(c->device));
                gl_stream_plan_t mine = sp;
                mine.self = g;
                std::vector<const uint64_t*> own;
                for (uint32_t w = 0; w < n_waves; w++)
                    for (uint32_t j = sp.group_width * (w * G + g); j < std::min(n_cols, sp.group_width * (w * G + g + 1)); j++) own.push_back(cols[j]);
                DevBuf stage;
                stage.ensure(stage_words);
                Tree* t = trees[g].get();
                coset_stream_impl(c, &mine, own.data(), input_is_coeffs, peer_bufs.data(), stage.p, t->leaves.p, t->digests.p, t->d_cap.p, t->cap.data());
            });
        if (all_ok && !streamed)
            phase([&] {   // B: iNTT + LDE of the column slice; every coset's rows go to their owners
                CUDA_CHECK(cudaSetDevice(c->device));
                const uint32_t n_cosets = 1u << rate_bits;
                const uint32_t first_coset = rate_bits ? h_bitrev((uint32_t)(((uint64_t)g * n_cosets / G) % n_cosets), rate_bits) : 0;
                lde_scatter_impl(c, nullptr, cols + plan.col_offsets[g], 0, plan.col_counts[g], log_n, rate_bits, input_is_coeffs, peer_leaves.data(), G,
                                 leaf_pitch, plan.col_offsets[g], trees[g]->coeffs.p, plan.pitches[g], first_coset, (int)g);
            });
        barrier.arrive_and_wait();               // every rank's shipments have landed (lde_scatter_impl returns after its last copy)
        all_ok = true;
        for (uint32_t q = 0; q < G; q++) all_ok = all_ok && rcs[q] == GL_OK;
        if (all_ok && !streamed)
            phase([&] {   // C: hash the own leaf range down to this rank's slice of the cap
                CUDA_CHECK(cudaSetDevice(c->device));
                Tree* t = trees[g].get();
                reset_stages(c, GL_STAGE_LEAF_HASH, GL_N_STAGES);
                record(c, GL_STAGE_LEAF_HASH);
                merkle_build(c, t->leaves.p, rows_per_rank, n_cols, leaf_pitch, local_cap_height, t->digests.p, t->d_cap.p,
                             &c->launches[GL_STAGE_LEAF_HASH], &c->launches[GL_STAGE_TREE], c->ev[GL_STAGE_TREE]);
                record(c, GL_STAGE_D2H);
                CUDA_CHECK(cudaMemcpyAsync(t->cap.data(), t->d_cap.p, 32ULL << local_cap_height, cudaMemcpyDeviceToHost, c->stream));
                read_stages(c, GL_STAGE_LEAF_HASH, GL_STAGE_D2H);
            });
        barrier.arrive_and_wait();               // nobody releases a leaf buffer a peer may still be copying into
    };

    // workers wait at a gate until every thread exists: if one cannot be started, the others leave without touching a barrier
    std::mutex gate_mu;
    std::condition_variable gate_cv;
    int gate = 0;   // 0 wait, 1 go, -1 cancel
    auto gated_worker = [&](uint32_t g) {
        {
            std::unique_lock<std::mutex> lk(gate_mu);
            gate_cv.wait(lk, [&] { return gate != 0; });
            if (gate < 0) return;
        }
        worker(g);
    };
    std::vector<std::thread> threads;
    bool started = true;
    try {
        for (uint32_t g = 1; g < G; g++) threads.emplace_back(gated_worker, g);
    } catch (...) {
        started = false;
    }
    {
        std::lock_guard<std::mutex> lk(gate_mu);
        gate = started ? 1 : -1;
    }
    gate_cv.notify_all();
    if (started) worker(0);
    for (auto& t : threads) t.join();
    if (!started) return fail0(GL_ERR_OOM, "could not start the worker threads");

    int rc = GL_OK;
    for (uint32_t g = 0; g < G && rc == GL_OK; g++) rc = rcs[g];
    if (rc != GL_OK) {
        for (uint32_t g = 0; g < G; g++) {
            std::lock_guard<std::mutex> lk(ctxs[g]->mu);
            cudaSetDevice(ctxs[g]->device);
            trees[g].reset();
        }
        if (rcs[0] == GL_OK) {   // report through the first context what a peer said
            for (uint32_t g = 1; g < G; g++)
                if (rcs[g] != GL_OK) { std::string m; { std::lock_guard<std::mutex> lk(ctxs[g]->mu); m = ctxs[g]->err; } fail0(rcs[g], m); break; }
        }
        return rc;
    }
    // rank q owns cap entries [q * 2^h / G, (q + 1) * 2^h / G)
    for (uint32_t g = 0; g < G; g++) {
        memcpy(out_cap + (size_t)g * (4ULL << local_cap_height), trees[g]->cap.data(), 32ULL << local_cap_height);
        std::lock_guard<std::mutex> lk(ctxs[g]->mu);
        out_trees[g] = ctxs[g]->trees.put(ctxs[g], std::move(trees[g]));
    }
    return GL_OK;
}

int gl_tree_info(gl_ctx* c, gl_handle h, gl_tree_info_t* out) {
    GL_API_BEGIN(c)
    if (!out) GL_THROW(GL_ERR_INVALID, "out is NULL");
    Tree* t = c->trees.get(h);
    out->n_leaves = t->n_leaves; out->leaf_len = t->leaf_len; out->cap_height = t->cap_height;
    out->degree_log = t->degree_log; out->rate_bits = t->rate_bits; out->has_coeffs = t->has_coeffs; out->pitch = t->pitch;
    return GL_OK;
    GL_API_END(c)
}

int gl_tree_get(gl_ctx* c, gl_handle h, uint64_t leaf_index, uint64_t* out_row) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(h);
    if (leaf_index >= t->n_leaves || !out_row) GL_THROW(GL_ERR_INVALID, "leaf index out of range");
    copy_row(c, t, leaf_index, out_row);
    return GL_OK;
    GL_API_END(c)
}

int gl_tree_get_lde_values(gl_ctx* c, gl_handle h, uint64_t index, uint64_t step, uint64_t* out_row) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(h);
    if (!out_row) GL_THROW(GL_ERR_INVALID, "out_row is NULL");
    if (step != 0 && index > (t->n_leaves - 1) / step) GL_THROW(GL_ERR_INVALID, "index * step out of range");   // also rules out a wrapped product
    uint64_t i = index * step;
    copy_row(c, t, h_bitrev((uint32_t)i, log2_exact(t->n_leaves)), out_row);
    return GL_OK;
    GL_API_END(c)
}

namespace {
// MerkleTree::get + MerkleTree::prove for n indices: one gather kernel, at most two device->host copies
void open_batch_impl(gl_ctx* c, Tree* t, const uint64_t* leaf_indices, uint32_t n, uint64_t* out_rows, uint64_t* out_siblings) {
    if (n == 0) return;
    if (!leaf_indices) GL_THROW(GL_ERR_INVALID, "leaf_indices is NULL");
    for (uint32_t q = 0; q < n; q++)
        if (leaf_indices[q] >= t->n_leaves) GL_THROW(GL_ERR_INVALID, "leaf index out of range");
    const uint32_t log_sub = log2_exact(t->n_leaves) - t->cap_height;
    const size_t row_words = out_rows ? (size_t)n * t->leaf_len : 0, sib_words = out_siblings ? (size_t)n * log_sub * 4 : 0;
    c->scratch.ensure(n + row_words + sib_words + 1);
    uint64_t* d_idx = c->scratch.p;
    uint64_t* d_rows = d_idx + n;
    uint64_t* d_sib = d_rows + row_words;
    CUDA_CHECK(cudaMemcpyAsync(d_idx, leaf_indices, 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    const uint64_t total = (uint64_t)n * (t->leaf_len + 4 * log_sub);
    if (total && (row_words || sib_words)) {
        merkle::open_batch_kernel<<<(uint32_t)((total + 255) / 256), 256, 0, c->stream>>>(
            t->leaves.p, t->pitch, t->leaf_len, t->digests.p, log_sub, d_idx, n, row_words ? d_rows : nullptr, sib_words ? d_sib : nullptr);
        CUDA_CHECK(cudaGetLastError());
    }
    if (row_words) CUDA_CHECK(cudaMemcpyAsync(out_rows, d_rows, 8 * row_words, cudaMemcpyDeviceToHost, c->stream));
    if (sib_words) CUDA_CHECK(cudaMemcpyAsync(out_siblings, d_sib, 8 * sib_words, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
}
}  // namespace

int gl_tree_prove(gl_ctx* c, gl_handle h, uint64_t leaf_index, uint64_t* out_siblings) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(h);
    if (leaf_index >= t->n_leaves) GL_THROW(GL_ERR_INVALID, "leaf index out of range");
    uint32_t log_sub = log2_exact(t->n_leaves) - t->cap_height;
    if (!out_siblings && log_sub) GL_THROW(GL_ERR_INVALID, "out_siblings is NULL");   /* an empty proof needs no buffer */
    open_batch_impl(c, t, &leaf_index, 1, nullptr, out_siblings);                      /* one gather + one copy, not one copy per level */
    return GL_OK;
    GL_API_END(c)
}

int gl_tree_open_batch(gl_ctx* c, gl_handle h, const uint64_t* leaf_indices, uint32_t n, uint64_t* out_rows, uint64_t* out_siblings) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(h);
    open_batch_impl(c, t, leaf_indices, n, out_rows, out_siblings);
    return GL_OK;
    GL_API_END(c)
}

int gl_tree_read(gl_ctx* c, gl_handle h, int part, uint64_t* out) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(h);
    if (!out) GL_THROW(GL_ERR_INVALID, "out is NULL");
    switch (part) {
        case GL_PART_COEFFS: {
            if (!t->has_coeffs) GL_THROW(GL_ERR_INVALID, "tree has no coefficients");
            uint64_t N = 1ULL << t->degree_log;
            c->scratch.ensure(N * t->leaf_len);
            dim3 tb(32, 8), tg((uint32_t)((N + 31) / 32), (t->leaf_len + 31) / 32);
            ntt::transpose_out_kernel<<<tg, tb, 0, c->stream>>>(t->coeffs.p, t->pitch, c->scratch.p, N, t->leaf_len, N);
            CUDA_CHECK(cudaGetLastError());
            CUDA_CHECK(cudaMemcpyAsync(out, c->scratch.p, N * t->leaf_len * 8, cudaMemcpyDeviceToHost, c->stream));
            break;
        }
        case GL_PART_LEAVES:
            if (t->leaf_len)
                CUDA_CHECK(cudaMemcpy2DAsync(out, (size_t)t->leaf_len * 8, t->leaves.p, (size_t)t->pitch * 8, (size_t)t->leaf_len * 8,
                                             t->n_leaves, cudaMemcpyDeviceToHost, c->stream));
            break;
        case GL_PART_DIGESTS:
            if (t->n_digests()) CUDA_CHECK(cudaMemcpyAsync(out, t->digests.p, t->n_digests() * 32, cudaMemcpyDeviceToHost, c->stream));
            break;
        case GL_PART_CAP: memcpy(out, t->cap.data(), t->cap.size() * 8); break;
        default: GL_THROW(GL_ERR_INVALID, "unknown part %d", part);
    }
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_tree_free(gl_ctx* c, gl_handle h) {
    GL_API_BEGIN(c)
    c->trees.drop(c, h);
    return GL_OK;
    GL_API_END(c)
}

// ------------------------------------------------------------------------------------------------ FRI
int gl_fri_begin(gl_ctx* c, const uint64_t* coeffs_ext, const uint64_t* values_ext, uint64_t len, uint32_t rate_bits,
                 uint32_t cap_height, gl_handle* out_fri) {
    GL_API_BEGIN(c)
    if (!coeffs_ext || !values_ext || !out_fri) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (len == 0 || (len & (len - 1)) || len > (1ULL << 31)) GL_THROW(GL_ERR_INVALID, "len must be a power of two");
    auto f = std::make_unique<Fri>(len, rate_bits, cap_height);
    CUDA_CHECK(cudaMemcpyAsync(f->coeffs.p, coeffs_ext, 16 * len, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(f->tmp.p, values_ext, 16 * len, cudaMemcpyHostToDevice, c->stream));
    fri::canon_kernel<<<(uint32_t)((2 * len + 255) / 256), 256, 0, c->stream>>>(f->coeffs.p, 2 * len);
    CUDA_CHECK(cudaGetLastError());
    uint32_t bits = log2_exact(len);
    fri::bitrev_gather_ext_kernel<<<(uint32_t)((len + 255) / 256), 256, 0, c->stream>>>(
        reinterpret_cast<const ulonglong2*>(f->tmp.p), reinterpret_cast<ulonglong2*>(f->values.p), bits);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    *out_fri = c->fris.put(c, std::move(f));
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_commit_layer(gl_ctx* c, gl_handle fh, uint32_t arity_bits, uint64_t* out_leaves, uint64_t* out_digests, uint64_t* out_cap,
                        gl_handle* out_tree) {
    GL_API_BEGIN(c)
    Fri* f = c->fris.get(fh);
    if (!out_cap) GL_THROW(GL_ERR_INVALID, "out_cap is NULL");
    uint64_t arity = 1ULL << arity_bits;
    if (arity > f->len) GL_THROW(GL_ERR_INVALID, "arity larger than the codeword");
    uint64_t n_leaves = f->len >> arity_bits;
    uint32_t leaf_len = (uint32_t)(2 * arity);
    if ((1ULL << f->cap_height) > n_leaves) GL_THROW(GL_ERR_INVALID, "cap_height should be at most log2(leaves.len())");
    const uint32_t pitch = round_up(leaf_len, 8);
    auto t = std::make_unique<Tree>(n_leaves, leaf_len, pitch, f->cap_height);
    // bit-reversed values chunked by arity ARE the leaves (flatten = the [a0,a1] interleaving already in memory)
    if (pitch == leaf_len) {
        CUDA_CHECK(cudaMemcpyAsync(t->leaves.p, f->values.p, 16 * f->len, cudaMemcpyDeviceToDevice, c->stream));
    } else {
        CUDA_CHECK(cudaMemcpy2DAsync(t->leaves.p, (size_t)pitch * 8, f->values.p, (size_t)leaf_len * 8, (size_t)leaf_len * 8, n_leaves,
                                     cudaMemcpyDeviceToDevice, c->stream));
    }
    merkle_build(c, t->leaves.p, n_leaves, leaf_len, pitch, f->cap_height, t->digests.p, t->d_cap.p, nullptr, nullptr, nullptr);
    if (out_leaves)
        CUDA_CHECK(cudaMemcpy2DAsync(out_leaves, (size_t)leaf_len * 8, t->leaves.p, (size_t)pitch * 8, (size_t)leaf_len * 8, n_leaves,
                                     cudaMemcpyDeviceToHost, c->stream));
    finish_tree(c, std::move(t), out_digests, out_cap, out_tree);
    f->last_arity_bits = arity_bits;
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_fold(gl_ctx* c, gl_handle fh, const uint64_t beta[2]) {
    GL_API_BEGIN(c)
    Fri* f = c->fris.get(fh);
    if (!beta) GL_THROW(GL_ERR_INVALID, "beta is NULL");
    if (f->last_arity_bits == 0) GL_THROW(GL_ERR_INVALID, "gl_fri_fold without a preceding gl_fri_commit_layer");
    NvtxRange nv("fold codewords in the commitment phase");
    const uint32_t arity_bits = f->last_arity_bits;   // upstream folds by the arity of the layer it just committed
    f->last_arity_bits = 0;
    uint64_t arity = 1ULL << arity_bits;
    if (arity > f->len) GL_THROW(GL_ERR_INVALID, "arity larger than the codeword");
    uint64_t n_out = f->len >> arity_bits;
    fri::fold_kernel<<<(uint32_t)((n_out + 127) / 128), 128, 0, c->stream>>>(
        reinterpret_cast<const ulonglong2*>(f->coeffs.p), reinterpret_cast<ulonglong2*>(f->tmp.p), (uint32_t)n_out, (uint32_t)arity,
        gl::canon(beta[0]), gl::canon(beta[1]));
    CUDA_CHECK(cudaGetLastError());
    std::swap(f->coeffs.p, f->tmp.p);
    std::swap(f->coeffs.words, f->tmp.words);
    f->len = n_out;
    f->shift = gl::h_pow(f->shift, arity);
    // values <- coset_fft(coeffs, shift), kept in bit-reversed (in-place DIF) order
    uint32_t log_len = log2_exact(n_out);
    run_ntt(c, f->coeffs.p, 2, f->values.p, 2, 2, log_len, false, get_coset_table(c, f->shift, log_len), 2, nullptr);
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_final_poly(gl_ctx* c, gl_handle fh, uint64_t* out, uint64_t* out_len) {
    GL_API_BEGIN(c)
    Fri* f = c->fris.get(fh);
    uint64_t n = f->len >> f->rate_bits;
    if (out_len) *out_len = n;
    if (out && n) CUDA_CHECK(cudaMemcpyAsync(out, f->coeffs.p, 16 * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_end(gl_ctx* c, gl_handle fh) {
    GL_API_BEGIN(c)
    c->fris.drop(c, fh);
    return GL_OK;
    GL_API_END(c)
}

// ------------------------------------------------------------------------------------------------ prove_openings (front half)
namespace {
struct HExt { uint64_t a0, a1; };
HExt h_ext_mul(HExt a, HExt b) {   // F_p[X]/(X^2 - 7)
    uint64_t m11 = gl::h_mul(a.a1, b.a1);
    HExt r;
    r.a0 = (uint64_t)(((unsigned __int128)gl::h_mul(a.a0, b.a0) + gl::h_mul(m11, 7)) % gl::P);
    r.a1 = (uint64_t)(((unsigned __int128)gl::h_mul(a.a0, b.a1) + gl::h_mul(a.a1, b.a0)) % gl::P);
    return r;
}
}  // namespace

int gl_openings_begin(gl_ctx* c, uint32_t log_n, gl_handle* out) {
    GL_API_BEGIN(c)
    if (!out) GL_THROW(GL_ERR_INVALID, "out_openings is NULL");
    if (log_n > 30) GL_THROW(GL_ERR_UNSUPPORTED, "log_n = %u > 30", log_n);
    auto o = std::make_unique<Openings>();
    o->log_n = log_n;
    const uint64_t n = 1ULL << log_n;
    o->final_poly.ensure(2 * n);
    o->comp.ensure(2 * n);
    CUDA_CHECK(cudaMemsetAsync(o->final_poly.p, 0, 16 * n, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    *out = c->openings.put(c, std::move(o));
    return GL_OK;
    GL_API_END(c)
}

int gl_openings_add_batch(gl_ctx* c, gl_handle oh, const gl_handle* batches, const uint32_t* columns, uint32_t n_polys,
                          const uint64_t alpha[2], const uint64_t point[2], uint64_t* out_quotient) {
    GL_API_BEGIN(c)
    Openings* o = c->openings.get(oh);
    if (!alpha || !point || (n_polys && (!batches || !columns))) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    const uint32_t n = 1u << o->log_n;
    std::vector<openings::PolyRef> refs(n_polys);
    std::vector<uint64_t> pw(2 * (size_t)n_polys);
    const HExt al = {gl::canon(alpha[0]), gl::canon(alpha[1])};
    HExt cur = {1, 0};
    for (uint32_t j = 0; j < n_polys; j++) {
        Tree* t = c->trees.get(batches[j]);
        if (!t->has_coeffs) GL_THROW(GL_ERR_INVALID, "polynomial %u: the tree has no coefficients", j);
        if (t->degree_log != o->log_n) GL_THROW(GL_ERR_INVALID, "Polynomial degrees inconsistent (polynomial %u has degree_log %u, expected %u)",
                                                j, t->degree_log, o->log_n);
        if (columns[j] >= t->leaf_len) GL_THROW(GL_ERR_INVALID, "polynomial %u: column %u out of range", j, columns[j]);
        refs[j] = {t->coeffs.p, t->pitch, columns[j]};
        pw[2 * j] = cur.a0; pw[2 * j + 1] = cur.a1;
        cur = h_ext_mul(cur, al);
    }
    // cur = alpha^n_polys: what shift_poly multiplies the running final_poly by
    if (n_polys) {
        static_assert(sizeof(openings::PolyRef) == 16, "PolyRef is two words");
        o->refs.ensure(2 * (size_t)n_polys);
        o->pw.ensure(2 * (size_t)n_polys);
        CUDA_CHECK(cudaMemcpyAsync(o->refs.p, refs.data(), 16 * (size_t)n_polys, cudaMemcpyHostToDevice, c->stream));
        CUDA_CHECK(cudaMemcpyAsync(o->pw.p, pw.data(), 16 * (size_t)n_polys, cudaMemcpyHostToDevice, c->stream));
        openings::reduce_polys_base_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(
            reinterpret_cast<const openings::PolyRef*>(o->refs.p), reinterpret_cast<const ulonglong2*>(o->pw.p), n_polys, n,
            reinterpret_cast<ulonglong2*>(o->comp.p));
        CUDA_CHECK(cudaGetLastError());
    } else {
        CUDA_CHECK(cudaMemsetAsync(o->comp.p, 0, 16 * (size_t)n, c->stream));
    }
    const uint32_t threads = n < 1024 ? n : 1024;
    openings::divide_by_linear_kernel<<<1, threads, 0, c->stream>>>(reinterpret_cast<ulonglong2*>(o->comp.p), n, gl::canon(point[0]),
                                                                    gl::canon(point[1]));
    CUDA_CHECK(cudaGetLastError());
    openings::shift_add_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(reinterpret_cast<ulonglong2*>(o->final_poly.p),
                                                                      reinterpret_cast<const ulonglong2*>(o->comp.p), n, cur.a0, cur.a1);
    CUDA_CHECK(cudaGetLastError());
    if (out_quotient) CUDA_CHECK(cudaMemcpyAsync(out_quotient, o->comp.p, 16 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));   // refs / pw are host vectors of this call
    return GL_OK;
    GL_API_END(c)
}

int gl_openings_final_poly(gl_ctx* c, gl_handle oh, uint64_t* out) {
    GL_API_BEGIN(c)
    Openings* o = c->openings.get(oh);
    if (!out) GL_THROW(GL_ERR_INVALID, "out is NULL");
    CUDA_CHECK(cudaMemcpyAsync(out, o->final_poly.p, 16ULL << o->log_n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_openings_lde(gl_ctx* c, gl_handle oh, uint32_t rate_bits, uint32_t cap_height, gl_handle* out_fri) {
    GL_API_BEGIN(c)
    Openings* o = c->openings.get(oh);
    if (!out_fri) GL_THROW(GL_ERR_INVALID, "out_fri is NULL");
    if (o->log_n + rate_bits > 31) GL_THROW(GL_ERR_UNSUPPORTED, "log_n + rate_bits = %u > 31", o->log_n + rate_bits);
    const uint64_t n = 1ULL << o->log_n, len = n << rate_bits;
    auto f = std::make_unique<Fri>(len, rate_bits, cap_height);
    // final_poly.lde(rate_bits): zero-padded coefficients; values = coset_fft(shift 7), kept bit-reversed (in-place DIF order)
    CUDA_CHECK(cudaMemsetAsync(f->coeffs.p, 0, 16 * len, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(f->coeffs.p, o->final_poly.p, 16 * n, cudaMemcpyDeviceToDevice, c->stream));
    const uint32_t log_len = o->log_n + rate_bits;
    if (log_len == 0) {
        CUDA_CHECK(cudaMemcpyAsync(f->values.p, f->coeffs.p, 16, cudaMemcpyDeviceToDevice, c->stream));
    } else {
        run_ntt(c, f->coeffs.p, 2, f->values.p, 2, 2, log_len, false, get_coset_table(c, gl::COSET_SHIFT, log_len), 2, nullptr);
    }
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    *out_fri = c->fris.put(c, std::move(f));
    return GL_OK;
    GL_API_END(c)
}

int gl_openings_end(gl_ctx* c, gl_handle oh) {
    GL_API_BEGIN(c)
    c->openings.drop(c, oh);
    return GL_OK;
    GL_API_END(c)
}

// ------------------------------------------------------------------------------------------------ OpeningSet::new
int gl_batch_eval(gl_ctx* c, gl_handle batch, const uint64_t* points_ext, uint32_t n_points, uint64_t* out_values_ext) {
    GL_API_BEGIN(c)
    Tree* t = c->trees.get(batch);
    if (!t->has_coeffs) GL_THROW(GL_ERR_INVALID, "tree has no coefficients");
    if (!points_ext || !out_values_ext) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_points == 0) GL_THROW(GL_ERR_INVALID, "n_points must be at least 1");
    if (n_points > 2) GL_THROW(GL_ERR_UNSUPPORTED, "n_points = %u > 2", n_points);
    openings::EvalPoints pts{};
    for (uint32_t p = 0; p < n_points; p++) {
        HExt z = {gl::canon(points_ext[2 * p]), gl::canon(points_ext[2 * p + 1])};
        for (uint32_t b = 0; b < 32; b++) {
            pts.z2k[p][b][0] = z.a0; pts.z2k[p][b][1] = z.a1;
            z = h_ext_mul(z, z);
        }
    }
    const uint64_t N = 1ULL << t->degree_log;
    const uint32_t sub_rows = (uint32_t)std::min<uint64_t>(N, openings::EVAL_SUB);
    const uint32_t col_tiles = (t->leaf_len + openings::EVAL_THREADS - 1) / openings::EVAL_THREADS;
    const uint32_t wc = (t->leaf_len + col_tiles - 1) / col_tiles;
    const uint32_t lanes = std::min(openings::EVAL_THREADS / wc, sub_rows);
    const uint32_t threads = round_up(lanes * wc, 32);
    uint32_t n_parts = (uint32_t)(N / sub_rows);   // row CTAs: a power of two, at most EVAL_MAX_PARTS / col_tiles
    while (n_parts > 1 && n_parts * col_tiles > openings::EVAL_MAX_PARTS) n_parts >>= 1;
    const uint32_t subs = (uint32_t)(N / sub_rows / n_parts);
    const uint32_t n_out = n_points * t->leaf_len;
    c->scratch.ensure(2 * (size_t)n_out * (n_parts + 1));
    ulonglong2* partial = reinterpret_cast<ulonglong2*>(c->scratch.p);
    ulonglong2* d_out = partial + (size_t)n_out * n_parts;
    const dim3 grid(n_parts, col_tiles);
    if (n_points == 1)
        openings::batch_eval_partial_kernel<1><<<grid, threads, 0, c->stream>>>(t->coeffs.p, t->pitch, t->leaf_len, wc, lanes, sub_rows, subs,
                                                                                 pts, partial);
    else
        openings::batch_eval_partial_kernel<2><<<grid, threads, 0, c->stream>>>(t->coeffs.p, t->pitch, t->leaf_len, wc, lanes, sub_rows, subs,
                                                                                 pts, partial);
    CUDA_CHECK(cudaGetLastError());
    openings::batch_eval_reduce_kernel<<<(n_out + 31) / 32, dim3(32, 32), 0, c->stream>>>(partial, n_parts, n_out, d_out);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(out_values_ext, d_out, 16 * (size_t)n_out, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_read(gl_ctx* c, gl_handle fh, uint64_t* out_coeffs, uint64_t* out_values, uint64_t* out_len) {
    GL_API_BEGIN(c)
    Fri* f = c->fris.get(fh);
    if (out_len) *out_len = f->len;
    if (out_coeffs) CUDA_CHECK(cudaMemcpyAsync(out_coeffs, f->coeffs.p, 16 * f->len, cudaMemcpyDeviceToHost, c->stream));
    if (out_values) CUDA_CHECK(cudaMemcpyAsync(out_values, f->values.p, 16 * f->len, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

// ------------------------------------------------------------------------------------------------ gates / quotient (§8f ranks 3-4)
namespace {
// wires / constraints per gate kind (param as documented in include/gl_commit.h); -1 for a bad kind or parameter
int gate_wires(int kind, uint32_t param) {
    const uint32_t lo = param & 0xFF, hi = param >> 8;
    switch (kind) {
        case GL_GATE_POSEIDON2: return gates::P2_NUM_WIRES;
        case GL_GATE_U32_ARITHMETIC: return param >= 1 && param <= 3 ? (int)((gates::U32_ROUTED + gates::U32_LIMBS) * param) : -1;
        case GL_GATE_U32_ADD_MANY: return lo >= 1 && lo <= 24 && hi >= 1 && (lo + 3 + 18) * hi <= 135 ? (int)((lo + 3 + 18) * hi) : -1;
        case GL_GATE_U32_SUBTRACTION: return param >= 1 && param <= 6 ? (int)(21 * param) : -1;
        case GL_GATE_U32_RANGE_CHECK: return param >= 1 && param <= 7 ? (int)(17 * param) : -1;
        case GL_GATE_U32_INTERLEAVE: return param >= 1 && param <= 3 ? (int)(34 * param) : -1;
        case GL_GATE_UNINTERLEAVE_TO_U32:
        case GL_GATE_UNINTERLEAVE_TO_B32: return param >= 1 && param <= 2 ? (int)(67 * param) : -1;
        case GL_GATE_COMPARISON: {
            if (lo < 1 || lo > 63 || hi < 1 || hi > lo) return -1;
            const uint32_t cb = (lo + hi - 1) / hi;
            return cb <= 6 && 4 + 5 * hi + cb + 1 <= 135 ? (int)(4 + 5 * hi + cb + 1) : -1;
        }
        case GL_GATE_NOOP: return param == 0 ? 0 : -1;
        case GL_GATE_CONSTANT: return param >= 1 && param <= 8 ? (int)param : -1;
        case GL_GATE_PUBLIC_INPUT: return param == 0 ? 4 : -1;
        case GL_GATE_ARITHMETIC: return param >= 1 && param <= 33 ? (int)(4 * param) : -1;
        case GL_GATE_BASE_SUM: return lo >= 1 && 1 + lo <= 135 && hi >= 2 && hi <= 16 ? (int)(1 + lo) : -1;
        case GL_GATE_POSEIDON: return param == 0 ? gates::P2_NUM_WIRES : -1;
        case GL_GATE_EXPONENTIATION: return param >= 1 && param <= 66 ? (int)(2 + 2 * param) : -1;
        case GL_GATE_RANDOM_ACCESS: {   // bits | num_copies << 8 | num_extra_constants << 16
            const uint32_t copies = hi & 0xFF, extras = param >> 16;
            if (lo < 1 || lo > 6 || copies < 1) return -1;
            const uint32_t nw = ((2u + (1u << lo)) + lo) * copies + extras;
            return nw <= 135 ? (int)nw : -1;
        }
        default: return -1;
    }
}
int gate_constraints(int kind, uint32_t param) {
    if (gate_wires(kind, param) < 0) return -1;
    const uint32_t lo = param & 0xFF, hi = param >> 8;
    switch (kind) {
        case GL_GATE_POSEIDON2: return gates::P2_NUM_CONSTRAINTS;
        case GL_GATE_U32_ARITHMETIC: return (int)((4 + gates::U32_LIMBS) * param);
        case GL_GATE_U32_ADD_MANY: return (int)(21 * hi);
        case GL_GATE_U32_SUBTRACTION: return (int)(19 * param);
        case GL_GATE_U32_RANGE_CHECK: return (int)(17 * param);
        case GL_GATE_U32_INTERLEAVE: return (int)(34 * param);
        case GL_GATE_UNINTERLEAVE_TO_U32:
        case GL_GATE_UNINTERLEAVE_TO_B32: return (int)(67 * param);
        case GL_GATE_COMPARISON: return (int)(2 + 5 * hi + 1 + ((lo + hi - 1) / hi + 1) + 2);
        case GL_GATE_NOOP: return 0;
        case GL_GATE_CONSTANT: return (int)param;
        case GL_GATE_PUBLIC_INPUT: return 4;
        case GL_GATE_ARITHMETIC: return (int)param;
        case GL_GATE_POSEIDON: return gates::P2_NUM_CONSTRAINTS;
        case GL_GATE_EXPONENTIATION: return (int)(param + 1);
        case GL_GATE_RANDOM_ACCESS: return (int)((lo + 2) * (hi & 0xFF) + (param >> 16));
        default: return (int)(1 + lo);   // GL_GATE_BASE_SUM
    }
}
int gate_constants(int kind, uint32_t param) {
    if (gate_wires(kind, param) < 0) return -1;
    switch (kind) {
        case GL_GATE_CONSTANT: return (int)param;
        case GL_GATE_ARITHMETIC: return 2;
        case GL_GATE_RANDOM_ACCESS: return (int)(param >> 16);
        default: return 0;
    }
}
void check_gate(int kind, uint32_t param) {
    if (kind < GL_GATE_POSEIDON2 || kind > GL_GATE_RANDOM_ACCESS || (kind > GL_GATE_BASE_SUM && kind < GL_GATE_POSEIDON))
        GL_THROW(GL_ERR_INVALID, "unknown gate kind %d", kind);
    if (gate_wires(kind, param) < 0) GL_THROW(GL_ERR_INVALID, "gate kind %d: parameter %u out of range (see include/gl_commit.h)", kind, param);
}
// the entry points without gate constants / public-inputs hash refuse the gates that read them
void check_gate_without_constants(int kind, uint32_t param, const char* entry) {
    check_gate(kind, param);
    if (gate_constants(kind, param) > 0 || kind == GL_GATE_PUBLIC_INPUT)
        GL_THROW(GL_ERR_INVALID, "gate kind %d reads gate constants or the public-inputs hash: use %s", kind, entry);
}

// gate constraints of host rows on the device: out [n_rows][num_constraints]; consts [n_rows][gate_constants] or NULL when that is 0
void eval_rows(gl_ctx* c, int kind, uint32_t param, const uint64_t* rows, const uint64_t* consts, const uint64_t* pi_hash, uint64_t n_rows,
               uint64_t* out) {
    const uint32_t nw = (uint32_t)gate_wires(kind, param), nc = (uint32_t)gate_constraints(kind, param), nk = (uint32_t)gate_constants(kind, param);
    if (n_rows == 0 || nc == 0) return;
    c->scratch.ensure(n_rows * (nw + nk + nc));
    uint64_t* d_rows = c->scratch.p;
    uint64_t* d_consts = d_rows + n_rows * nw;
    uint64_t* d_out = d_consts + n_rows * nk;
    gates::PiHash pi{};
    for (int i = 0; i < 4 && pi_hash; i++) pi.w[i] = gl::canon(pi_hash[i]);
    CUDA_CHECK(cudaMemcpyAsync(d_rows, rows, n_rows * nw * 8, cudaMemcpyHostToDevice, c->stream));
    if (nk) CUDA_CHECK(cudaMemcpyAsync(d_consts, consts, n_rows * nk * 8, cudaMemcpyHostToDevice, c->stream));
    gates::gate_constraints_kernel<<<(uint32_t)((n_rows + 127) / 128), 128, 0, c->stream>>>(kind, param, d_rows, nw, n_rows, nc, d_consts, nk, pi,
                                                                                             d_out);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(out, d_out, n_rows * nc * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
}

// alpha_k^(offset + i), i < nc, for every challenge: [n_ch][nc] (a few hundred host multiplies per gate)
void alpha_powers(const uint64_t* alphas, uint32_t n_ch, uint32_t offset, uint32_t nc, uint64_t* out) {
    for (uint32_t k = 0; k < n_ch; k++) {
        const uint64_t al = gl::canon(alphas[k]);
        uint64_t cur = gl::h_pow(al, offset);
        for (uint32_t i = 0; i < nc; i++) { out[(size_t)k * nc + i] = cur; cur = gl::h_mul(cur, al); }
    }
}

void launch_gate_quotient(gl_ctx* c, const gates::QuotientArgs& a) {
    // PoseidonGate has its own instances: the shared switch keeps the registers (and CTAs per SM) it has without it
    static void (*const kernels[2][4])(gates::QuotientArgs) = {
        {gates::gate_quotient_kernel<1>, gates::gate_quotient_kernel<2>, gates::gate_quotient_kernel<3>, gates::gate_quotient_kernel<4>},
        {gates::gate_quotient_kernel<1, true>, gates::gate_quotient_kernel<2, true>, gates::gate_quotient_kernel<3, true>,
         gates::gate_quotient_kernel<4, true>}};
    const uint32_t grid = (uint32_t)((a.n_rows + 127) / 128);
    const size_t smem = (size_t)a.n_challenges * a.n_constraints * 8;
    kernels[a.kind == GL_GATE_POSEIDON][std::min(a.n_challenges, 4u) - 1]<<<grid, 128, smem, c->stream>>>(a);
    CUDA_CHECK(cudaGetLastError());
}

// gl_poseidon2_gate_witness / gl_poseidon_gate_witness: inputs [n][13] -> out_rows [n][135], kernel time in aux_ms
void gate_witness(gl_ctx* c, const uint64_t* inputs, uint64_t n, uint64_t* out_rows,
                  void (*kernel)(const uint64_t*, uint64_t, uint64_t*, uint32_t)) {
    if ((!inputs || !out_rows) && n) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n == 0) return;
    c->scratch.ensure(n * (13 + gates::P2_NUM_WIRES));
    uint64_t* d_in = c->scratch.p;
    uint64_t* d_out = d_in + n * 13;
    CUDA_CHECK(cudaMemcpyAsync(d_in, inputs, n * 13 * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev[0], c->stream));
    kernel<<<(uint32_t)((n + 127) / 128), 128, 0, c->stream>>>(d_in, n, d_out, gates::P2_NUM_WIRES);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaEventRecord(c->ev[1], c->stream));
    CUDA_CHECK(cudaMemcpyAsync(out_rows, d_out, n * gates::P2_NUM_WIRES * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    CUDA_CHECK(cudaEventElapsedTime(&c->aux_ms, c->ev[0], c->ev[1]));
}
}  // namespace

int gl_gate_num_wires(int kind, uint32_t param) { return gate_wires(kind, param); }
int gl_gate_num_constraints(int kind, uint32_t param) { return gate_constraints(kind, param); }
int gl_gate_num_constants(int kind, uint32_t param) { return gate_constants(kind, param); }

int gl_gate_eval_rows(gl_ctx* c, int kind, uint32_t param, const uint64_t* rows, uint64_t n_rows, uint64_t* out) {
    GL_API_BEGIN(c)
    check_gate_without_constants(kind, param, "gl_gate_eval_rows_with_constants");
    if ((!rows || !out) && n_rows) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    eval_rows(c, kind, param, rows, nullptr, nullptr, n_rows, out);
    return GL_OK;
    GL_API_END(c)
}

int gl_gate_eval_rows_with_constants(gl_ctx* c, int kind, uint32_t param, const uint64_t* rows, const uint64_t* consts,
                                     const uint64_t public_inputs_hash[4], uint64_t n_rows, uint64_t* out) {
    GL_API_BEGIN(c)
    check_gate(kind, param);
    if (!public_inputs_hash) GL_THROW(GL_ERR_INVALID, "public_inputs_hash is NULL");
    if ((!rows || !out || (!consts && gate_constants(kind, param) > 0)) && n_rows) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    eval_rows(c, kind, param, rows, consts, public_inputs_hash, n_rows, out);
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_begin(gl_ctx* c, gl_handle wires_batch, uint32_t n_challenges, gl_handle* out_q) {
    GL_API_BEGIN(c)
    if (!out_q) GL_THROW(GL_ERR_INVALID, "out_quotient is NULL");
    if (n_challenges == 0 || n_challenges > (uint32_t)gates::MAX_CHALLENGES) GL_THROW(GL_ERR_INVALID, "n_challenges must be 1..%d", gates::MAX_CHALLENGES);
    Tree* t = c->trees.get(wires_batch);
    auto q = std::make_unique<Quotient>();
    q->wires = wires_batch; q->n_rows = t->n_leaves; q->n_challenges = n_challenges;
    q->acc.ensure(q->n_rows * n_challenges);
    q->powers.ensure((size_t)gates::MAX_CHALLENGES * gates::MAX_CONSTRAINTS);
    CUDA_CHECK(cudaMemsetAsync(q->acc.p, 0, q->n_rows * n_challenges * 8, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    *out_q = c->quotients.put(c, std::move(q));
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_add_gate(gl_ctx* c, gl_handle qh, int kind, uint32_t param, const uint64_t* alphas, uint32_t constraint_offset,
                         gl_handle filter_batch, uint32_t filter_col) {
    GL_API_BEGIN(c)
    Quotient* q = c->quotients.get(qh);
    check_gate_without_constants(kind, param, "gl_quotient_add_gates");
    if (!alphas) GL_THROW(GL_ERR_INVALID, "alphas is NULL");
    Tree* t = c->trees.get(q->wires);
    const uint32_t nw = (uint32_t)gate_wires(kind, param), nc = (uint32_t)gate_constraints(kind, param);
    if (t->leaf_len < nw) GL_THROW(GL_ERR_INVALID, "the wires batch has %u columns, the gate needs %u", t->leaf_len, nw);
    if (nc > (uint32_t)gates::MAX_CONSTRAINTS) GL_THROW(GL_ERR_UNSUPPORTED, "too many constraints");
    gates::QuotientArgs a{};
    a.rows = t->leaves.p; a.pitch = t->pitch; a.n_rows = q->n_rows; a.acc = q->acc.p; a.powers = q->powers.p;
    a.n_constraints = nc; a.n_challenges = q->n_challenges; a.kind = (uint32_t)kind; a.param = param;
    if (filter_batch) {
        Tree* f = c->trees.get(filter_batch);
        if (f->n_leaves != q->n_rows) GL_THROW(GL_ERR_INVALID, "filter batch has %llu rows, the wires batch %llu", (unsigned long long)f->n_leaves, (unsigned long long)q->n_rows);
        if (filter_col >= f->leaf_len) GL_THROW(GL_ERR_INVALID, "filter column %u out of range", filter_col);
        a.filter = f->leaves.p; a.filter_pitch = f->pitch; a.filter_col = filter_col; a.filter_mode = gates::FILTER_COLUMN;
    }
    c->aux_ms = 0;
    if (nc == 0) return GL_OK;   // NoopGate
    std::vector<uint64_t> pw((size_t)q->n_challenges * nc);
    alpha_powers(alphas, q->n_challenges, constraint_offset, nc, pw.data());
    CUDA_CHECK(cudaMemcpyAsync(q->powers.p, pw.data(), pw.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev[0], c->stream));
    launch_gate_quotient(c, a);
    CUDA_CHECK(cudaEventRecord(c->ev[1], c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));   // pw is a host vector of this call
    CUDA_CHECK(cudaEventElapsedTime(&c->aux_ms, c->ev[0], c->ev[1]));
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_add_gates(gl_ctx* c, gl_handle qh, const int* kinds, const uint32_t* params, uint32_t n_gates, const uint32_t* selector_indices,
                          const uint32_t* groups, uint32_t num_selectors, uint32_t num_lookup_selectors, gl_handle constants_sigmas,
                          uint32_t num_constants, const uint64_t public_inputs_hash[4], const uint64_t* alphas, uint32_t constraint_offset) {
    GL_API_BEGIN(c)
    Quotient* q = c->quotients.get(qh);
    if (!kinds || !params || !selector_indices || !groups || !public_inputs_hash || !alphas) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_gates == 0) GL_THROW(GL_ERR_INVALID, "No gates?");
    Tree* tw = c->trees.get(q->wires);
    Tree* tc = c->trees.get(constants_sigmas);
    if (tc->n_leaves != tw->n_leaves || tc->degree_log != tw->degree_log || tc->rate_bits != tw->rate_bits)
        GL_THROW(GL_ERR_INVALID, "Polynomial degrees inconsistent (the constants/sigmas batch must share the wires batch's rows, degree and rate_bits)");
    if (num_constants > tc->leaf_len) GL_THROW(GL_ERR_INVALID, "num_constants %u exceeds the constants/sigmas batch's %u columns", num_constants, tc->leaf_len);
    const uint32_t const_col0 = num_selectors + num_lookup_selectors;
    // every gate is checked before the first launch: a refused call leaves the accumulator as it was
    uint32_t max_nc = 0;
    for (uint32_t i = 0; i < n_gates; i++) {
        check_gate(kinds[i], params[i]);
        const uint32_t nw = (uint32_t)gate_wires(kinds[i], params[i]), nc = (uint32_t)gate_constraints(kinds[i], params[i]);
        const uint32_t s = selector_indices[i];
        if (s >= num_selectors) GL_THROW(GL_ERR_INVALID, "gate %u: selector index %u >= num_selectors %u", i, s, num_selectors);
        if (groups[2 * s] > groups[2 * s + 1] || groups[2 * s + 1] > n_gates)
            GL_THROW(GL_ERR_INVALID, "selector group %u = [%u, %u) is not a range of the %u gates", s, groups[2 * s], groups[2 * s + 1], n_gates);
        if (i < groups[2 * s] || i >= groups[2 * s + 1])
            GL_THROW(GL_ERR_INVALID, "gate %u is outside its selector group %u = [%u, %u)", i, s, groups[2 * s], groups[2 * s + 1]);
        if (const_col0 + (uint32_t)gate_constants(kinds[i], params[i]) > num_constants)
            GL_THROW(GL_ERR_INVALID, "gate %u: %u selector columns + %u gate constants exceed num_constants %u", i, const_col0,
                     (uint32_t)gate_constants(kinds[i], params[i]), num_constants);
        if (tw->leaf_len < nw) GL_THROW(GL_ERR_INVALID, "gate %u: the wires batch has %u columns, the gate needs %u", i, tw->leaf_len, nw);
        if (nc > (uint32_t)gates::MAX_CONSTRAINTS) GL_THROW(GL_ERR_UNSUPPORTED, "gate %u: too many constraints", i);
        max_nc = std::max(max_nc, nc);
    }
    const uint32_t n_ch = q->n_challenges;
    c->aux_ms = 0;
    if (max_nc == 0) return GL_OK;   // only NoopGates
    // every gate's constraints start at alpha^offset (evaluate_gate_constraints_base_batch sums them into one constraint vector)
    std::vector<uint64_t> pw((size_t)n_ch * max_nc);
    alpha_powers(alphas, n_ch, constraint_offset, max_nc, pw.data());
    gates::QuotientArgs a{};
    a.rows = tw->leaves.p; a.pitch = tw->pitch; a.n_rows = q->n_rows; a.acc = q->acc.p; a.n_challenges = n_ch;
    a.filter = tc->leaves.p; a.filter_pitch = tc->pitch; a.filter_mode = gates::FILTER_SELECTOR;
    a.many_selectors = num_selectors > 1; a.const_col0 = const_col0;
    for (int j = 0; j < 4; j++) a.pi.w[j] = gl::canon(public_inputs_hash[j]);
    // one [n_ch][nc] table per gate (the kernel reads its table with row stride nc), uploaded in one copy
    std::vector<uint64_t> host;
    std::vector<size_t> table_at(n_gates);
    for (uint32_t i = 0; i < n_gates; i++) {
        const uint32_t nc = (uint32_t)gate_constraints(kinds[i], params[i]);
        table_at[i] = host.size();
        for (uint32_t k = 0; k < n_ch; k++) host.insert(host.end(), pw.begin() + (size_t)k * max_nc, pw.begin() + (size_t)k * max_nc + nc);
    }
    c->scratch.ensure(host.size());
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, host.data(), host.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev[0], c->stream));
    for (uint32_t i = 0; i < n_gates; i++) {
        const uint32_t nc = (uint32_t)gate_constraints(kinds[i], params[i]), s = selector_indices[i];
        if (nc == 0) continue;   // NoopGate
        a.kind = (uint32_t)kinds[i]; a.param = params[i]; a.n_constraints = nc; a.powers = c->scratch.p + table_at[i];
        a.gate_index = i; a.filter_col = s; a.group_start = groups[2 * s]; a.group_end = groups[2 * s + 1];
        launch_gate_quotient(c, a);
    }
    CUDA_CHECK(cudaEventRecord(c->ev[1], c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));   // `host` is a vector of this call
    CUDA_CHECK(cudaEventElapsedTime(&c->aux_ms, c->ev[0], c->ev[1]));
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_add_permutation(gl_ctx* c, gl_handle qh, gl_handle sigmas_batch, uint32_t sigma_col0, gl_handle zs_batch, uint32_t n_routed,
                                uint32_t degree, const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, const uint64_t* alphas) {
    GL_API_BEGIN(c)
    Quotient* q = c->quotients.get(qh);
    if (!k_is || !betas || !gammas || !alphas) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_routed == 0 || degree == 0) GL_THROW(GL_ERR_INVALID, "n_routed and degree must be positive");
    Tree* tw = c->trees.get(q->wires);
    Tree* ts = c->trees.get(sigmas_batch);
    Tree* tz = c->trees.get(zs_batch);
    const uint32_t n_ch = q->n_challenges, n_chunks = (n_routed + degree - 1) / degree, n_terms = n_ch * (1 + n_chunks);
    if (!tw->has_coeffs || tw->rate_bits > 6) GL_THROW(GL_ERR_UNSUPPORTED, "the wires batch must be a PolynomialBatch commit with rate_bits <= 6");
    for (Tree* t : {ts, tz})
        if (t->n_leaves != tw->n_leaves || t->degree_log != tw->degree_log || t->rate_bits != tw->rate_bits)
            GL_THROW(GL_ERR_INVALID, "Polynomial degrees inconsistent (the sigma / Z batches must share the wires batch's degree and rate_bits)");
    if (tw->leaf_len < n_routed) GL_THROW(GL_ERR_INVALID, "the wires batch has %u columns, %u routed wires requested", tw->leaf_len, n_routed);
    if (sigma_col0 + n_routed > ts->leaf_len) GL_THROW(GL_ERR_INVALID, "sigma columns [%u, %u) out of range", sigma_col0, sigma_col0 + n_routed);
    if (tz->leaf_len != n_ch * n_chunks) GL_THROW(GL_ERR_INVALID, "the Z / partial-products batch must have n_challenges * ceil(n_routed / degree) = %u columns", n_ch * n_chunks);
    if (n_terms > (uint32_t)gates::MAX_CONSTRAINTS) GL_THROW(GL_ERR_UNSUPPORTED, "too many permutation terms");
    const uint32_t log_n = tw->degree_log, r = tw->rate_bits, bits = log_n + r;
    perm::VanishArgs a{};
    a.wires = tw->leaves.p; a.wires_pitch = tw->pitch;
    a.sigmas = ts->leaves.p; a.sigmas_pitch = ts->pitch; a.sigma_col0 = sigma_col0;
    a.zs = tz->leaves.p; a.zs_pitch = tz->pitch;
    a.W = get_roots(c, bits);
    a.acc = q->acc.p;
    a.log_n = log_n; a.rate_bits = r; a.n_routed = n_routed; a.degree = degree; a.n_chunks = n_chunks; a.n_ch = n_ch;
    a.n_inv = gl::h_inv(((uint64_t)1 << log_n) % gl::P);
    {
        const uint64_t gN = gl::h_pow(gl::COSET_SHIFT, 1ULL << log_n), wr = gl::h_root_of_unity(r);
        uint64_t cur = gN;
        for (uint32_t j = 0; j < (1u << r); j++) { a.zh[j] = cur - 1; cur = gl::h_mul(cur, wr); }
    }
    std::vector<uint64_t> host(n_routed + (size_t)n_ch * n_terms);
    for (uint32_t j = 0; j < n_routed; j++) host[j] = gl::canon(k_is[j]);
    for (uint32_t k = 0; k < n_ch; k++) {
        a.beta[k] = gl::canon(betas[k]); a.gamma[k] = gl::canon(gammas[k]);
        const uint64_t al = gl::canon(alphas[k]);
        uint64_t cur = 1;
        for (uint32_t t = 0; t < n_terms; t++) { host[n_routed + (size_t)k * n_terms + t] = cur; cur = gl::h_mul(cur, al); }
    }
    c->scratch.ensure(host.size());
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, host.data(), host.size() * 8, cudaMemcpyHostToDevice, c->stream));
    a.k_is = c->scratch.p;
    a.powers = c->scratch.p + n_routed;
    const uint32_t grid = (uint32_t)((q->n_rows + 127) / 128);
    const size_t smem = (size_t)n_ch * n_terms * 8;
    CUDA_CHECK(cudaEventRecord(c->ev[0], c->stream));
    switch (n_ch) {
        case 1: perm::vanishing_perm_kernel<1><<<grid, 128, smem, c->stream>>>(a); break;
        case 2: perm::vanishing_perm_kernel<2><<<grid, 128, smem, c->stream>>>(a); break;
        case 3: perm::vanishing_perm_kernel<3><<<grid, 128, smem, c->stream>>>(a); break;
        default: perm::vanishing_perm_kernel<4><<<grid, 128, smem, c->stream>>>(a); break;
    }
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaEventRecord(c->ev[1], c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    CUDA_CHECK(cudaEventElapsedTime(&c->aux_ms, c->ev[0], c->ev[1]));
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_read(gl_ctx* c, gl_handle qh, uint64_t* out) {
    GL_API_BEGIN(c)
    Quotient* q = c->quotients.get(qh);
    if (!out) GL_THROW(GL_ERR_INVALID, "out is NULL");
    CUDA_CHECK(cudaMemcpyAsync(out, q->acc.p, q->n_rows * q->n_challenges * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_quotient_commit(gl_ctx* c, gl_handle qh, uint32_t cap_height, uint64_t* out_cap, gl_handle* out_batch) {
    GL_API_BEGIN(c)
    Quotient* q = c->quotients.get(qh);
    Tree* t = c->trees.get(q->wires);
    if (!out_cap) GL_THROW(GL_ERR_INVALID, "out_cap is NULL");
    const uint32_t log_n = t->degree_log, r = t->rate_bits, bits = log_n + r, n_ch = q->n_challenges;
    if (!t->has_coeffs) GL_THROW(GL_ERR_INVALID, "the wires batch is not a PolynomialBatch commit");
    if (bits < 3) GL_THROW(GL_ERR_UNSUPPORTED, "quotient domain smaller than 8 points");
    const uint64_t N = 1ULL << log_n, R = 1ULL << bits;
    const uint32_t pitch = 4, n_chunks = 1u << r;
    // Z_H(g w_R^i)^-1 for i mod 2^r, and shift^-j (host: 2^r inversions; the tables are filled on the device)
    std::vector<uint64_t> zh(1u << r);
    const uint64_t gN = gl::h_pow(gl::COSET_SHIFT, N), wr = gl::h_root_of_unity(r);
    uint64_t cur = gN;
    for (uint32_t j = 0; j < (1u << r); j++) { zh[j] = gl::h_inv(cur - 1); cur = gl::h_mul(cur, wr);   /* cur is a non-zero canonical element; Z_H != 0 on the coset */ }
    DevBuf vals, coeffs, tab, cols;
    vals.ensure(R * pitch); coeffs.ensure(R * pitch); tab.ensure(R + 8); cols.ensure((uint64_t)n_ch * R);
    uint64_t* d_zh = tab.p + R;
    CUDA_CHECK(cudaMemcpyAsync(d_zh, zh.data(), zh.size() * 8, cudaMemcpyHostToDevice, c->stream));
    gates::quotient_gather_kernel<<<(uint32_t)((R + 255) / 256), 256, 0, c->stream>>>(q->acc.p, vals.p, pitch, n_ch, bits, r, d_zh);
    CUDA_CHECK(cudaGetLastError());
    run_ntt(c, vals.p, pitch, coeffs.p, pitch, pitch, bits, true, nullptr, 4, nullptr);           // ifft: natural values -> natural coefficients
    {
        ntt::PowTable pt{};
        uint64_t sq = gl::h_inv(gl::COSET_SHIFT);
        for (uint32_t k = 0; k < 32; k++) { pt.g2k[k] = sq; sq = gl::h_mul(sq, sq); }
        ntt::powers_kernel<<<(uint32_t)((R + 255) / 256), 256, 0, c->stream>>>(tab.p, R, pt);
        CUDA_CHECK(cudaGetLastError());
    }
    gates::quotient_chunks_kernel<<<(uint32_t)((R + 255) / 256), 256, 0, c->stream>>>(coeffs.p, pitch, n_ch, log_n, r, tab.p, cols.p);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaStreamSynchronize(c->stream));   // zh is a host vector of this call
    return commit_impl(c, nullptr, cols.p, N, n_ch * n_chunks, log_n, r, cap_height, 1, nullptr, nullptr, nullptr, out_cap, out_batch);
    GL_API_END(c)
}

int gl_quotient_end(gl_ctx* c, gl_handle qh) {
    GL_API_BEGIN(c)
    c->quotients.drop(c, qh);
    return GL_OK;
    GL_API_END(c)
}

int gl_ctx_aux_ms(gl_ctx* c, float* out_ms) {
    if (!c || !out_ms) return GL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(c->mu);
    *out_ms = c->aux_ms;
    return GL_OK;
}

int gl_poseidon2_gate_witness(gl_ctx* c, const uint64_t* inputs, uint64_t n, uint64_t* out_rows) {
    GL_API_BEGIN(c)
    gate_witness(c, inputs, n, out_rows, gates::poseidon2_witness_kernel);
    return GL_OK;
    GL_API_END(c)
}

int gl_poseidon_gate_witness(gl_ctx* c, const uint64_t* inputs, uint64_t n, uint64_t* out_rows) {
    GL_API_BEGIN(c)
    gate_witness(c, inputs, n, out_rows, gates::poseidon_witness_kernel);
    return GL_OK;
    GL_API_END(c)
}

int gl_partial_products(gl_ctx* c, const uint64_t* const* wire_cols, const uint64_t* const* sigma_cols, uint32_t n_routed, uint32_t log_n,
                        const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, uint32_t n_ch, uint32_t degree, uint64_t* out_cols) {
    GL_API_BEGIN(c)
    if (!wire_cols || !sigma_cols || !k_is || !betas || !gammas || !out_cols) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_routed == 0 || degree == 0) GL_THROW(GL_ERR_INVALID, "n_routed and degree must be positive");
    if (n_ch == 0 || n_ch > 4) GL_THROW(GL_ERR_INVALID, "n_challenges must be 1..4");
    if (log_n > 28) GL_THROW(GL_ERR_UNSUPPORTED, "log_n = %u > 28", log_n);
    const uint32_t n_chunks = (n_routed + degree - 1) / degree;
    if (n_chunks > (uint32_t)perm::MAX_CHUNKS) GL_THROW(GL_ERR_UNSUPPORTED, "more than %d chunks (n_routed / degree)", perm::MAX_CHUNKS);
    for (uint32_t j = 0; j < n_routed; j++)
        if (!wire_cols[j] || !sigma_cols[j]) GL_THROW(GL_ERR_INVALID, "column %u is NULL", j);
    const uint64_t N = 1ULL << log_n;
    const uint32_t pitch = round_up(n_routed, 8);
    // layout of the scratch: wires [N][pitch] | sigmas [N][pitch] | xs [N] | k_is | q [n_ch][N][n_chunks] | out [n_ch*n_chunks][N]
    const size_t w_words = N * pitch, q_words = (size_t)n_ch * N * n_chunks;
    c->in_stage.ensure(2 * N * n_routed);
    c->scratch.ensure(2 * w_words + N + round_up(n_routed, 8) + 2 * q_words);
    uint64_t* d_w = c->scratch.p;
    uint64_t* d_s = d_w + w_words;
    uint64_t* d_x = d_s + w_words;
    uint64_t* d_k = d_x + N;
    uint64_t* d_q = d_k + round_up(n_routed, 8);
    uint64_t* d_out = d_q + q_words;
    for (uint32_t j = 0; j < n_routed; j++) {
        CUDA_CHECK(cudaMemcpyAsync(c->in_stage.p + (uint64_t)j * N, wire_cols[j], N * 8, cudaMemcpyHostToDevice, c->stream));
        CUDA_CHECK(cudaMemcpyAsync(c->in_stage.p + (uint64_t)(n_routed + j) * N, sigma_cols[j], N * 8, cudaMemcpyHostToDevice, c->stream));
    }
    std::vector<uint64_t> kk(n_routed);
    for (uint32_t j = 0; j < n_routed; j++) kk[j] = gl::canon(k_is[j]);
    CUDA_CHECK(cudaMemcpyAsync(d_k, kk.data(), n_routed * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev[0], c->stream));
    dim3 tb(32, 8), tg((uint32_t)((N + 31) / 32), (pitch + 31) / 32);
    ntt::transpose_in_kernel<<<tg, tb, 0, c->stream>>>(c->in_stage.p, N, d_w, pitch, pitch, n_routed, N);
    ntt::transpose_in_kernel<<<tg, tb, 0, c->stream>>>(c->in_stage.p + (uint64_t)n_routed * N, N, d_s, pitch, pitch, n_routed, N);
    CUDA_CHECK(cudaGetLastError());
    {
        ntt::PowTable pt{};
        uint64_t sq = gl::h_root_of_unity(log_n);
        for (uint32_t k = 0; k < 32; k++) { pt.g2k[k] = sq; sq = gl::h_mul(sq, sq); }
        ntt::powers_kernel<<<(uint32_t)((N + 255) / 256), 256, 0, c->stream>>>(d_x, N, pt);
        CUDA_CHECK(cudaGetLastError());
    }
    perm::Args a{};
    a.wires = d_w; a.sigmas = d_s; a.k_is = d_k; a.xs = d_x; a.q = d_q; a.out = d_out;
    for (uint32_t k = 0; k < n_ch; k++) { a.beta[k] = gl::canon(betas[k]); a.gamma[k] = gl::canon(gammas[k]); }
    a.n = (uint32_t)N; a.pitch = pitch; a.n_routed = n_routed; a.degree = degree; a.n_chunks = n_chunks; a.n_ch = n_ch;
    perm::chunk_quotients_kernel<<<dim3((uint32_t)((N + 127) / 128), n_ch), 128, 0, c->stream>>>(a);
    CUDA_CHECK(cudaGetLastError());
    perm::running_product_kernel<<<n_ch, 1024, 0, c->stream>>>(a);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaEventRecord(c->ev[1], c->stream));
    CUDA_CHECK(cudaMemcpyAsync(out_cols, d_out, q_words * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    CUDA_CHECK(cudaEventElapsedTime(&c->aux_ms, c->ev[0], c->ev[1]));
    return GL_OK;
    GL_API_END(c)
}

int gl_poseidon_permute(gl_ctx* c, uint64_t* states, uint64_t n) {
    GL_API_BEGIN(c)
    if (!states && n) GL_THROW(GL_ERR_INVALID, "states is NULL");
    if (n == 0) return GL_OK;
    c->scratch.ensure(12 * n);
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, states, 96 * n, cudaMemcpyHostToDevice, c->stream));
    merkle::permute_kernel<<<(uint32_t)((n + 127) / 128), 128, 0, c->stream>>>(c->scratch.p, n);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(states, c->scratch.p, 96 * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_poseidon_absorb(gl_ctx* c, uint64_t state[12], const uint64_t* groups, uint32_t n_groups) {
    GL_API_BEGIN(c)
    if (!state || (!groups && n_groups)) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if (n_groups == 0) return GL_OK;
    c->scratch.ensure(12 + 8ULL * n_groups);
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, state, 96, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p + 12, groups, 64ULL * n_groups, cudaMemcpyHostToDevice, c->stream));
    merkle::sponge_absorb_kernel<<<1, 32, 0, c->stream>>>(c->scratch.p, c->scratch.p + 12, n_groups);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(state, c->scratch.p, 96, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

// element-wise field primitives exactly as the kernels use them (unit tests of the carry logic on adversarial words)
__global__ void field_op_kernel(int op, const uint64_t* __restrict__ a, const uint64_t* __restrict__ b, uint64_t* __restrict__ out,
                                uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t x = a[i], y = b[i], r = 0;
    switch (op & ~GL_FOP_RAW) {
        case GL_FOP_MUL: r = gl::mul(x, y); break;
        case GL_FOP_ADD_ANY: r = gl::add_any(x, y); break;
        case GL_FOP_SUB_ANY: r = gl::sub_any(x, y); break;
        case GL_FOP_MUL_2_24: r = gl::mul_2_24(x); break;
        case GL_FOP_MUL_2_48: r = gl::mul_2_48(x); break;
        case GL_FOP_MUL_2_72: r = gl::mul_2_72(x); break;
        case GL_FOP_SBOX7: {
            double lo, hi;
            poseidon::sbox7_limbs(x, lo, hi);
            // same read-out as the MDS layer: bias + positivity offset, then recombine (offsets are = 0 mod p)
            r = poseidon::recombine(__dadd_rn(lo, 4503599627370496.0 + 562949953552384.0), __dadd_rn(hi, 4503599627370496.0 + 562949953159168.0));
            break;
        }
        case GL_FOP_ADD_ANY_C: r = gl::add_any_c(x, gl::canon(y)); break;
        default: break;
    }
    out[i] = (op & GL_FOP_RAW) ? r : gl::canon(r);
}

int gl_field_op(gl_ctx* c, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint64_t n) {
    GL_API_BEGIN(c)
    if (!a || !b || !out) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    if ((op & ~GL_FOP_RAW) < 0 || (op & ~GL_FOP_RAW) > GL_FOP_ADD_ANY_C) GL_THROW(GL_ERR_INVALID, "unknown field op %d", op);
    if (n == 0) return GL_OK;
    c->scratch.ensure(3 * n);
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, a, 8 * n, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p + n, b, 8 * n, cudaMemcpyHostToDevice, c->stream));
    field_op_kernel<<<(uint32_t)((n + 127) / 128), 128, 0, c->stream>>>(op, c->scratch.p, c->scratch.p + n, c->scratch.p + 2 * n, n);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(out, c->scratch.p + 2 * n, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return GL_OK;
    GL_API_END(c)
}

int gl_fri_pow(gl_ctx* c, const uint64_t sponge_state[12], const uint64_t* input_buffer, uint32_t n_inputs, uint32_t min_leading_zeros,
               uint64_t* out_witness) {
    GL_API_BEGIN(c)
    if (!sponge_state || !out_witness || (n_inputs && !input_buffer)) GL_THROW(GL_ERR_INVALID, "NULL pointer");
    NvtxRange nv("find proof-of-work witness");
    if (n_inputs >= 8) GL_THROW(GL_ERR_INVALID, "input buffer must hold fewer than SPONGE_RATE = 8 elements");
    if (min_leading_zeros > 40) GL_THROW(GL_ERR_UNSUPPORTED, "min_leading_zeros = %u: search space too large", min_leading_zeros);
    uint64_t st[12];
    for (int i = 0; i < 12; i++) st[i] = gl::canon(sponge_state[i]);
    for (uint32_t i = 0; i < n_inputs; i++) st[i] = gl::canon(input_buffer[i]);
    c->scratch.ensure(16);
    unsigned long long* d_best = reinterpret_cast<unsigned long long*>(c->scratch.p + 12);
    const unsigned long long none = ~0ULL;
    CUDA_CHECK(cudaMemcpyAsync(c->scratch.p, st, sizeof st, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaMemcpyAsync(d_best, &none, 8, cudaMemcpyHostToDevice, c->stream));
    // windows grow geometrically from ~4x the expected number of tries; every candidate below a window was rejected
    uint64_t window = std::max<uint64_t>(1ULL << 16, 4ULL << min_leading_zeros);
    window = std::min<uint64_t>(window, 1ULL << 28);
    for (uint64_t base = 0;; base += window) {
        if (base >= gl::P) GL_THROW(GL_ERR_INVALID, "no proof-of-work witness exists");
        merkle::pow_grind_kernel<<<(uint32_t)((window + 127) / 128), 128, 0, c->stream>>>(c->scratch.p, n_inputs, min_leading_zeros, base,
                                                                                        window, d_best);
        CUDA_CHECK(cudaGetLastError());
        unsigned long long best = none;
        CUDA_CHECK(cudaMemcpyAsync(&best, d_best, 8, cudaMemcpyDeviceToHost, c->stream));
        CUDA_CHECK(cudaStreamSynchronize(c->stream));
        if (best != none) { *out_witness = best; break; }
    }
    return GL_OK;
    GL_API_END(c)
}

int gl_ctx_stage_times(gl_ctx* c, float* out_ms, uint32_t* out_launches) {
    if (!c || !out_ms) return GL_ERR_INVALID;
    std::lock_guard<std::mutex> lk(c->mu);
    memcpy(out_ms, c->stage_ms, sizeof c->stage_ms);
    if (out_launches) memcpy(out_launches, c->launches, sizeof c->launches);
    return GL_OK;
}

int gl_microbench(gl_ctx* c, int which, uint32_t iters, double* out_ops_per_s) {
    GL_API_BEGIN(c)
    if (!out_ops_per_s || iters == 0) GL_THROW(GL_ERR_INVALID, "bad arguments");
    const int threads = 256;
    const int blocks = c->sm_count * (which == 4 ? 4 : 8);
    c->scratch.ensure((size_t)threads * blocks);
    cudaEvent_t e0 = c->ev[0], e1 = c->ev[1];
    double ops = 0;
    for (int rep = 0; rep < 2; rep++) {   // first repetition warms up
        CUDA_CHECK(cudaEventRecord(e0, c->stream));
        switch (which) {
            case 0: microbench::imad_wide_kernel<<<blocks, threads, 0, c->stream>>>(c->scratch.p, iters, 0x9E3779B9u); break;
            case 1: microbench::alu_kernel<<<blocks, threads, 0, c->stream>>>(c->scratch.p, iters, 0x9E3779B9u); break;
            case 2: microbench::mixed_kernel<<<blocks, threads, 0, c->stream>>>(c->scratch.p, iters, 0x9E3779B9u); break;
            case 3: microbench::modmul_kernel<<<blocks, threads, 0, c->stream>>>(c->scratch.p, iters, 0x123456789ABCDEF1ULL); break;
            case 4: microbench::poseidon_kernel<<<blocks, threads, 0, c->stream>>>(c->scratch.p, iters); break;
            default: GL_THROW(GL_ERR_INVALID, "unknown microbenchmark %d", which);
        }
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaEventRecord(e1, c->stream));
        CUDA_CHECK(cudaStreamSynchronize(c->stream));
        float ms = 0;
        CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        double per_thread = which == 4 ? (double)iters : (which == 2 ? 2.0 : 1.0) * 4.0 * microbench::CHAINS * iters;
        ops = per_thread * threads * blocks / (ms * 1e-3);
    }
    *out_ops_per_s = ops;
    return GL_OK;
    GL_API_END(c)
}

void* gl_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void gl_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
