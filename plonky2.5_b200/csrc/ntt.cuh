// K1/K2/K3: batched Goldilocks NTT over a ROW-MAJOR matrix [rows][pitch] (one column = one polynomial).
//
// Replaces plonky2 field/src/fft.rs · fft_classic / ifft_with_options, field/src/polynomial/mod.rs · lde /
// coset_fft_with_options, and util/src/lib.rs · transpose + reverse_index_bits_in_place (SURVEY.md A.2-A.4);
// driven from /root/reference/src/p3/mod.rs:250,260 through PolynomialBatch::from_values / from_coeffs.
//
// Why row-major: the Merkle leaves are rows, so the LDE must END row-major with bit-reversed row order.  Keeping
// the matrix row-major through every pass means (i) every HBM access is a G-column segment of a row (32/64 B,
// sector aligned because pitch % 8 == 0) whatever row permutation a pass needs, (ii) an in-place decimation-in-
// frequency NTT leaves row p holding X[bitrev(p)] — exactly plonky2's leaf order — so the "transpose +
// reverse_index_bits" stage of the reference costs nothing here, and (iii) the iFFT's index reversal
// out[i] = b[(n-i) mod n] is just the store address of the last pass.
//
// One pass = a 2^a-point DIF NTT (a <= 10) on index bits [log_blk-a, log_blk) of every block of 2^log_blk rows,
// staged through shared memory in radix-8 register rounds (8-point DFTs whose roots are powers of two, i.e. shifts,
// then one table twiddle per element), followed (if lower bits remain) by the inter-pass twiddle
// w_{2^log_blk}^(o_lo * bitrev_a(l)) (four-step factorisation).  Round twiddles come from a 7*2^a/8-entry
// shared-memory table; all roots come from one table W[e] = w_N^e (e < N/2) held by the context.
#pragma once
#include "gl_field.cuh"

namespace ntt {

constexpr int MAX_PEERS = 16;

struct PassParams {
    const uint64_t* src;
    uint64_t* dst;
    uint32_t src_pitch, dst_pitch;   // words
    uint32_t log_n;                  // NTT size
    uint32_t log_blk;                // block size entering this pass (log_n for the first pass)
    uint32_t a;                      // stages done in this pass (>= 3)
    uint32_t ncg;                    // column groups (pitch / G)
    const uint64_t* W;               // w_N^e, e < max(N/2, 1), canonical
    const uint64_t* Wa;              // w_T^e, e < 7T/8 (T = 2^a), the upper eighths as -w_T^(e - T/2): round twiddles of this pass size
    const uint64_t* pre;             // coset pre-scale (first pass only): g^row, row < N, or nullptr
    uint32_t store_mode;             // 0: row p -> p ; 1: iFFT: row p -> (N - bitrev_n(p)) mod N ; 2: scatter to leaf owners
    uint64_t scale;                  // multiply at store when != 1 (1/N for the iFFT)
    // store_mode 2 (multi-GPU, last pass of a coset): row p of this coset is leaf row  scatter_row0 + p  of the global
    // leaf matrix; its owner is rank (row >> log_rows_per_peer) and the 8-column segment goes straight into that rank's
    // leaf buffer (peer pointer over NVLink, or local) at columns [scatter_col0, ...): the column->row exchange is
    // the NTT's own store, there is no all-to-all and no repacking.
    uint64_t* peer[MAX_PEERS];
    uint64_t scatter_row0;
    uint32_t log_rows_per_peer, scatter_col0, scatter_pitch, scatter_ncols;   // padding columns (>= ncols) are not stored
    // src_list != 0 (second-generation kernel, first pass only): column group cg is read from its OWN block peer[cg] = [N][G] (pitch
    // src_pitch == G) instead of columns [cg*G, (cg+1)*G) of src — the streamed coset plan evaluates the groups pulled from all peers
    // in one launch, straight from the separate blocks they arrived in
    uint32_t src_list;
};

__device__ __forceinline__ uint32_t ins3(uint32_t q, uint32_t sh, uint32_t e) {
    return ((q >> sh) << (sh + 3)) | (e << sh) | (q & ((1u << sh) - 1));
}
__device__ __forceinline__ uint32_t phys_row(uint32_t l) { return l + (l >> 3); }   // bank-conflict padding

__device__ __forceinline__ void addsub(uint64_t& u, uint64_t& v) {
    const uint64_t s = gl::add_any(u, v);
    v = gl::sub_any(u, v);
    u = s;
}

// In-place 8-point DIF with plonky2's power-of-two roots (w_8 = 2^120 = -2^24, w_4 = 2^48, w_8^3 = -2^72):
// on return x[e] = sum_j x_j w_8^(j * bitrev3(e)).  "any" in, "any" out; 24 add/sub + 5 shift-multiplies, no table.
__device__ __forceinline__ void dft8(uint64_t (&x)[8]) {
    uint64_t s;
    addsub(x[0], x[4]);
    s = gl::add_any(x[1], x[5]); x[5] = gl::mul_2_24(gl::sub_any(x[5], x[1])); x[1] = s;   // * w_8   = -2^24
    s = gl::add_any(x[2], x[6]); x[6] = gl::mul_2_48(gl::sub_any(x[2], x[6])); x[2] = s;   // * w_8^2 =  2^48
    s = gl::add_any(x[3], x[7]); x[7] = gl::mul_2_72(gl::sub_any(x[7], x[3])); x[3] = s;   // * w_8^3 = -2^72
#pragma unroll
    for (int h = 0; h < 8; h += 4) {
        addsub(x[h], x[h + 2]);
        s = gl::add_any(x[h + 1], x[h + 3]); x[h + 3] = gl::mul_2_48(gl::sub_any(x[h + 1], x[h + 3])); x[h + 1] = s;
    }
#pragma unroll
    for (int e = 0; e < 8; e += 2) addsub(x[e], x[e + 1]);
}

// One register round on the 8 elements of a thread: `nst` DIF stages on thread-local bits nst-1..0 (tile bit of local
// bit k is sh + k).  nst == 3 is a radix-8 step of a block of m = 2^(sh+3) tile rows: 8-point DFT, then element e is
// multiplied by w_m^(i * bitrev3(e)), i = position inside the sub-block (Wl[j] = w_T^j, j < 7T/8).  nst < 3 only
// happens with sh == 0, where every twiddle is a power of w_4.
__device__ __forceinline__ void radix8_round(uint64_t (&x)[8], const uint64_t* __restrict__ Wl, uint32_t a,
                                             uint32_t sh, uint32_t qlo, uint32_t nst) {
    if (nst == 3) {
        dft8(x);
        if (sh != 0) {
            const uint32_t step = qlo << (a - sh - 3);
#pragma unroll
            for (int e = 1; e < 8; e++) {
                const uint32_t k = ((e & 1) << 2) | (e & 2) | (e >> 2);
                x[e] = gl::mul(x[e], Wl[step * k]);
            }
        }
    } else if (nst == 2) {
#pragma unroll
        for (int h = 0; h < 8; h += 4) {
            addsub(x[h], x[h + 2]);
            const uint64_t s = gl::add_any(x[h + 1], x[h + 3]);
            x[h + 3] = gl::mul_2_48(gl::sub_any(x[h + 1], x[h + 3]));
            x[h + 1] = s;
            addsub(x[h], x[h + 1]);
            addsub(x[h + 2], x[h + 3]);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 8; e += 2) addsub(x[e], x[e + 1]);
    }
}

// A > 0: the pass size is a compile-time constant (round shifts, tile addressing and the round structure fold away);
// A == 0: generic (runtime p.a) — used for the 2-column FRI matrices.
template <int G, int A>
__global__ void __launch_bounds__(A ? (1 << A) * G / 8 : 1024, A ? ((1536 * 8 / ((1 << A) * G)) > 16 ? 16 : (1536 * 8 / ((1 << A) * G)) ? (1536 * 8 / ((1 << A) * G)) : 1) : 1)
ntt_pass_kernel(const PassParams p) {   // >= 48 resident warps per SM where the shape allows it
    extern __shared__ uint64_t sm[];
    const uint32_t a = A ? A : p.a, T = 1u << a;
    uint64_t* tile = sm;
    uint64_t* Wl = sm + (size_t)(T + (T >> 3)) * G;
    const uint32_t tid = threadIdx.x, nthr = blockDim.x;   // nthr = T*G/8
    const uint32_t c = tid % G, q = tid / G;
    const uint32_t cg = blockIdx.x % p.ncg, tile_id = blockIdx.x / p.ncg;
    const uint32_t b_lo = p.log_blk - a;
    const uint32_t o_lo = tile_id & ((1u << b_lo) - 1), o_hi = tile_id >> b_lo;
    const uint32_t row_base = (o_hi << p.log_blk) | o_lo;
    const uint32_t col = cg * G + c;

    // The tile's own loads go first: they are strided gathers from HBM and everything below waits for them, so the
    // round-twiddle staging (a contiguous, L2-resident table) and the pre-scale factors are fetched in their shadow.
    uint64_t x[8];
    uint32_t sh = a - 3;
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const uint64_t row = row_base | ((uint64_t)ins3(q, sh, e) << b_lo);
        x[e] = p.src[row * p.src_pitch + col];
    }
    // Wl[e] = w_T^e for e < 7T/8 (radix-8 twiddle exponents reach 7 * (T/8 - 1); the upper part is -w_T^(e - T/2)):
    // p.Wa is that table for this pass size, contiguous in global memory
    for (uint32_t e = tid; e < T - (T >> 3); e += nthr) Wl[e] = __ldg(p.Wa + e);
    if (p.pre != nullptr) {
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const uint64_t row = row_base | ((uint64_t)ins3(q, sh, e) << b_lo);
            x[e] = gl::mul(x[e], __ldg(p.pre + row));
        }
    }
    __syncthreads();   // Wl ready
    if (A) {
        // compile-time round structure: round r does min(3, A - 3r) stages at shift max(A - 3(r+1), 0)
        constexpr int ROUNDS = (A + 2) / 3;
#pragma unroll
        for (int r = 0; r < ROUNDS; r++) {
            constexpr int AA = A ? A : 3;
            const int done = 3 * r, left = AA - done;
            const uint32_t nst = left >= 3 ? 3 : left;
            const uint32_t shr = left >= 3 ? left - 3 : 0;
            if (r > 0) {
                const uint32_t shp = AA - 3 * r;   // shift of the previous round (>= 0 because r < ROUNDS)
#pragma unroll
                for (int e = 0; e < 8; e++) tile[(size_t)phys_row(ins3(q, shp, e)) * G + c] = x[e];
                __syncthreads();
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = tile[(size_t)phys_row(ins3(q, shr, e)) * G + c];
                if (r + 1 < ROUNDS) __syncthreads();   // the tile is rewritten by the next exchange
            }
            radix8_round(x, Wl, a, shr, q & ((1u << shr) - 1), nst);
            sh = shr;
        }
    } else {
        uint32_t remaining = a;
        while (true) {
            const uint32_t nst = remaining >= 3 ? 3 : remaining;
            radix8_round(x, Wl, a, sh, q & ((1u << sh) - 1), nst);
            remaining -= nst;
            if (remaining == 0) break;
#pragma unroll
            for (int e = 0; e < 8; e++) tile[(size_t)phys_row(ins3(q, sh, e)) * G + c] = x[e];
            __syncthreads();
            sh = remaining >= 3 ? remaining - 3 : 0;
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = tile[(size_t)phys_row(ins3(q, sh, e)) * G + c];
            __syncthreads();
        }
    }
    // sh is the shift of the last round: element e of this thread is tile row l = ins3(q, sh, e)
    const uint32_t N = 1u << p.log_n;
#pragma unroll
    for (int e = 0; e < 8; e++) {
        uint32_t l = ins3(q, sh, e);
        uint64_t v = x[e];
        if (b_lo) {
            // inter-pass twiddle w_{2^log_blk}^(o_lo * bitrev_a(l)), looked up in W (w_N^e, e < N/2)
            uint32_t ex = (o_lo * gl::bitrev32(l, a)) << (p.log_n - p.log_blk);
            uint64_t w;
            if (ex >= (N >> 1)) w = gl::P - p.W[ex - (N >> 1)];
            else w = p.W[ex];
            v = gl::mul(v, w);
        }
        if (p.scale != 1) v = gl::mul(v, p.scale);
        if (!b_lo) v = gl::canon(v);   // only what leaves the NTT is canonical; between passes any 64-bit representative will do
        uint32_t prow = row_base | (l << b_lo);
        if (p.store_mode == 2) {
            if (col >= p.scatter_ncols) continue;
            const uint64_t grow = p.scatter_row0 + prow;
            uint64_t* base = p.peer[grow >> p.log_rows_per_peer];
            base[(grow & ((1ULL << p.log_rows_per_peer) - 1)) * p.scatter_pitch + p.scatter_col0 + col] = v;
        } else {
            uint32_t drow = p.store_mode == 1 ? ((N - gl::bitrev32(prow, p.log_n)) & (N - 1)) : prow;
            p.dst[(uint64_t)drow * p.dst_pitch + col] = v;
        }
    }
}

// NTT sizes 1, 2, 4 (log_n < 3): direct O(N^2) evaluation, one thread per (output row, column).
// Produces the same in-place-DIF order (row p holds X[bitrev(p)]) / iFFT order as the pass kernel.
struct Scatter {   // see PassParams
    uint64_t* peer[MAX_PEERS];
    uint64_t row0;
    uint32_t log_rows_per_peer, col0, pitch, ncols;
    uint32_t self;   // index of the local buffer in peer[] (MAX_PEERS if unknown); host-side use only
};

__global__ void ntt_tiny_kernel(const uint64_t* __restrict__ src, uint64_t* __restrict__ dst, uint32_t src_pitch,
                                uint32_t dst_pitch, uint32_t n_cols, uint32_t log_n, uint64_t root, uint64_t g,
                                uint32_t store_mode, uint64_t scale, const Scatter sc) {
    const uint32_t N = 1u << log_n;
    uint32_t col = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t p = blockIdx.y;
    if (col >= n_cols) return;
    uint32_t k = gl::bitrev32(p, log_n);
    // X[k] = sum_j x_j g^j root^(jk)
    uint64_t wk = 1;
    for (uint32_t i = 0; i < k; i++) wk = gl::mulc(wk, root);
    uint64_t step = gl::mulc(wk, g), cur = 1, acc = 0;
    for (uint32_t j = 0; j < N; j++) {
        acc = gl::add(acc, gl::mulc(src[(uint64_t)j * src_pitch + col], cur));
        cur = gl::mulc(cur, step);
    }
    if (scale != 1) acc = gl::mulc(acc, scale);
    if (store_mode == 2) {
        if (col >= sc.ncols) return;
        const uint64_t grow = sc.row0 + p;
        sc.peer[grow >> sc.log_rows_per_peer][(grow & ((1ULL << sc.log_rows_per_peer) - 1)) * sc.pitch + sc.col0 + col] = acc;
        return;
    }
    uint32_t drow = store_mode == 1 ? ((N - k) & (N - 1)) : p;
    dst[(uint64_t)drow * dst_pitch + col] = acc;
}

// out[j] = g^j (canonical), j < n <= 2^32, from the table g2k[k] = g^(2^k)
struct PowTable { uint64_t g2k[32]; };
__global__ void powers_kernel(uint64_t* __restrict__ out, uint64_t n, const PowTable pt) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint64_t acc = 1;
#pragma unroll 1
    for (uint32_t k = 0, e = (uint32_t)j; e; k++, e >>= 1)
        if (e & 1) acc = gl::mul(acc, pt.g2k[k]);
    out[j] = gl::canon(acc);
}

// Column-major [n_cols][n_rows] (contiguous columns, as plonky2's Vec<PolynomialValues>) -> row-major
// [n_rows][pitch], canonicalising on the way.  32x32 tiles through shared memory.
__global__ void transpose_in_kernel(const uint64_t* __restrict__ src, uint64_t src_col_stride, uint64_t* __restrict__ dst,
                                    uint32_t pitch, uint32_t width, uint32_t n_cols, uint64_t n_rows) {
    // writes columns [0, width) of dst (row stride `pitch`): the n_cols source columns, zero beyond them
    __shared__ uint64_t t[32][33];
    uint64_t r0 = (uint64_t)blockIdx.x * 32;
    uint32_t c0 = blockIdx.y * 32;
    for (uint32_t i = threadIdx.y; i < 32; i += blockDim.y) {
        uint32_t c = c0 + i;
        uint64_t r = r0 + threadIdx.x;
        t[i][threadIdx.x] = (c < n_cols && r < n_rows) ? gl::canon(src[c * src_col_stride + r]) : 0;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.y; i < 32; i += blockDim.y) {
        uint64_t r = r0 + i;
        uint32_t c = c0 + threadIdx.x;
        if (r < n_rows && c < width) dst[r * pitch + c] = t[threadIdx.x][i];
    }
}

// Row-major [n_rows][pitch] -> column-major [n_cols][n_rows]
__global__ void transpose_out_kernel(const uint64_t* __restrict__ src, uint32_t pitch, uint64_t* __restrict__ dst,
                                     uint64_t dst_col_stride, uint32_t n_cols, uint64_t n_rows) {
    __shared__ uint64_t t[32][33];
    uint64_t r0 = (uint64_t)blockIdx.x * 32;
    uint32_t c0 = blockIdx.y * 32;
    for (uint32_t i = threadIdx.y; i < 32; i += blockDim.y) {
        uint64_t r = r0 + i;
        uint32_t c = c0 + threadIdx.x;
        t[i][threadIdx.x] = (r < n_rows && c < n_cols) ? src[r * pitch + c] : 0;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.y; i < 32; i += blockDim.y) {
        uint32_t c = c0 + i;
        uint64_t r = r0 + threadIdx.x;
        if (c < n_cols && r < n_rows) dst[c * dst_col_stride + r] = t[threadIdx.x][i];
    }
}

// Row-major [n_rows][src_pitch] -> row-major [n_rows][dst_pitch] (n_cols copied, canonicalised, padding zeroed);
// used when MerkleTree::new leaves arrive packed from the host and for multi-GPU repacking.
__global__ void repitch_kernel(const uint64_t* __restrict__ src, uint64_t src_pitch, uint64_t* __restrict__ dst,
                               uint32_t dst_pitch, uint32_t dst_col_off, uint32_t n_cols, uint64_t n_rows) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t r = i / n_cols;
    uint32_t c = (uint32_t)(i % n_cols);
    if (r < n_rows) dst[r * dst_pitch + dst_col_off + c] = gl::canon(src[r * src_pitch + c]);
}

}  // namespace ntt
