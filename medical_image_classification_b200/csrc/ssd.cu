// ssd.cu -- Mamba-2 SSD chunked scan (mamba_chunk_scan_combined), forward and backward, sm_100a.
//
// Replaces the un-vendored Triton kernels of mamba_ssm==2.2.2 that the reference calls at
// SSD/MedSSD.py:361-375 (semantics: SURVEY.md section 8(a) row a7).  Chunk-wise evaluation with
// chunk length Q (= chunk_size), per batch b, chunk c, head h (group g = h / (H/G)):
//
//   dt'_l  = clamp(softplus(dt_l + dt_bias_h))      cs_l = cumsum_{j<=l}(dt'_j A_h)   (within chunk)
//   CB     = C B^T                                  (Q x Q, per group)
//   Sloc   = sum_s exp(cs_Q - cs_s) dt'_s x_s (x) B_s            (P x N, per head)
//   Sin[c+1] = exp(cs_Q) Sin[c] + Sloc[c]                          (state passing)
//   y_l    = sum_{s<=l} CB[l,s] exp(cs_l - cs_s) dt'_s x_s + exp(cs_l) C_l Sin^T + D x_l
//
// Every contraction runs on the tensor cores through one CTA-level tile engine (TileMma below):
// 128x64x32 tiles, operands staged global -> registers -> shared with the decay / dt' factors
// applied on the way in, TF32 mma with the 3xTF32 split (hi*hi + hi*lo + lo*hi, fp32 accumulate)
// so that fp32 callers get fp32-accurate products (precision = 0), or a single TF32 pass
// (precision = 1: what the reference's tl.dot does on fp32 inputs).  Two interchangeable engines run the tiles: tcgen05.mma with
// TMEM accumulators (TcEngine, the default; UTCHMMA / LDTM in SASS) and warp-level mma.sync tiles (MmaEngine, HMMA in SASS).
// The backward is the exact adjoint of the chunked forward; it re-uses the forward's dt', cs,
// chunk-entry states and C B^T (workspace) and the forward output (for the "stable" d cs term).
#include <cstddef>
#include <cstdlib>

#include "common.cuh"

namespace b200 {
namespace ssd {

constexpr int BM = 128, BN = 64, BK = 32;
constexpr int NTHR = 256;
constexpr int LDA_KM = BM + 8, LDA_MK = BK + 4;
constexpr int LDB_KN = BN + 8, LDB_NK = BK + 4;
constexpr int A_FLOATS = (BK * LDA_KM > BM * LDA_MK) ? BK * LDA_KM : BM * LDA_MK;  // 4608
constexpr int B_FLOATS = (BK * LDB_KN > BN * LDB_NK) ? BK * LDB_KN : BN * LDB_NK;  // 2304
constexpr int MAXQ = 256;

// seq_idx (batch, L): packed variable-length rows; p == NULL is one sequence per row
struct Seq {
    const int32_t* p;
    int64_t s0, s1;
    __device__ __forceinline__ int at(int b, int l) const { return __ldg(p + b * s0 + (int64_t)l * s1); }
};

struct Dims {
    int batch, L, H, P, G, N, Q, nc, hpg;
    Seq seq;
};

// Masks of a packed row (seq_idx non-decreasing): with sid(l) = seq_idx[b][l], for chunk c of row b
//   intra-chunk term (l, s):       sid(l) == sid(s)
//   chunk-entry term at l:         sid(l) == seq_prev(c)   (the id at the previous chunk's last position, 0 before chunk 0)
//   chunk-state contribution of s: sid(s) == seq_end(c)    (the id at this chunk's last position)
//   state passing into chunk c+1:  seq_end(c) == seq_prev(c)
// The backward applies the same masks to the adjoint.  Each is a per-row or per-column factor of a contraction except the
// intra-chunk one, which the SEQ instantiations apply per element where the causal mask already is.
__device__ __forceinline__ int seq_prev(const Dims& d, int b, int c) { return c > 0 ? d.seq.at(b, c * d.Q - 1) : 0; }
__device__ __forceinline__ int seq_end(const Dims& d, int b, int c) { return d.seq.at(b, min((c + 1) * d.Q, d.L) - 1); }
// seq_idx of chunk c's position i (positions past the end of the row repeat the last id)
__device__ __forceinline__ int seq_at(const Dims& d, int b, int c, int i) { return d.seq.at(b, min(c * d.Q + i, d.L - 1)); }

struct Ws {  // views into the forward workspace
    float* dtp;     // [b][h][nc][Q]
    float* cs;      // [b][h][nc][Q]
    float* states;  // [b][nc][h][P][N]
    float* cb;      // [b][nc][g][Q][Q]
};

__host__ __device__ inline size_t ws_dt_floats(const Dims& d) { return (size_t)d.batch * d.H * d.nc * d.Q; }
__host__ __device__ inline size_t ws_state_floats(const Dims& d) { return (size_t)d.batch * d.nc * d.H * d.P * d.N; }
__host__ __device__ inline size_t ws_cb_floats(const Dims& d) { return (size_t)d.batch * d.nc * d.G * d.Q * d.Q; }

static Dims make_dims(const b200_ssd_fwd_params& p) {
    Dims d;
    d.batch = p.batch; d.L = p.seqlen; d.H = p.nheads; d.P = p.headdim; d.G = p.n_groups; d.N = p.dstate; d.Q = p.chunk_size;
    d.nc = (p.seqlen + p.chunk_size - 1) / p.chunk_size;
    d.hpg = p.nheads / p.n_groups;
    d.seq = Seq{p.seq_idx, p.seq_idx_stride[0], p.seq_idx_stride[1]};
    return d;
}
static Ws make_ws(float* base, const Dims& d) {
    Ws w;
    w.dtp = base;
    w.cs = w.dtp + ws_dt_floats(d);
    w.states = w.cs + ws_dt_floats(d);
    w.cb = w.states + ws_state_floats(d);
    return w;
}

// strided 4-D view (batch, L, head|group, inner)
template <typename T>
struct View4 {
    const T* p;
    int64_t s0, s1, s2, s3;
    __device__ __forceinline__ float at(int b, int l, int h, int i) const {
        return to_f32<T>(__ldg(p + b * s0 + l * s1 + h * s2 + i * s3));
    }
};
template <typename T> static View4<T> view4(const void* p, const int64_t* s) { return View4<T>{(const T*)p, s[0], s[1], s[2], s[3]}; }

// element strides of a gradient output (batch, L, head | group, p | n): the backward writes every gradient in the layout the caller
// asks for -- the layout of its primal in the models (sequence-contiguous channel-major storage), so no strided copy follows and
// the epilogue stores of a warp (32 consecutive sequence positions, one column) are contiguous
struct OutS {
    int64_t s0, s1, s2, s3;
    __device__ __forceinline__ size_t at(int b, int l, int h, int p) const { return (size_t)(b * s0 + (int64_t)l * s1 + h * s2 + p * s3); }
};
static OutS outs_of(const int64_t* s, int64_t d1, int64_t d2, int64_t d3) {   // all-zero strides = contiguous (batch, L, d2, d3)
    if (s[0] == 0 && s[1] == 0 && s[2] == 0 && s[3] == 0) return OutS{d1 * d2 * d3, d2 * d3, d3, 1};
    return OutS{s[0], s[1], s[2], s[3]};
}

// ---- tensor-core tile engine -----------------------------------------------------------------
__device__ __forceinline__ uint32_t tf32_rna(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

struct Acc {
    float v[2][4][4];  // [m16 block][n8 block][c0..c3] of this warp's 32x32 sub-tile
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int r = 0; r < 4; ++r) v[i][j][r] = 0.f;
    }
};

// ---- operand tiles: global -> registers (raw, 128-bit when possible) -> shared (transformed) ----------
// Logical tile [TI rows (m or n index i)][32 k].  KI = true: shared layout [k][i] (pitch TI+8) and the
// register tile is vectorised along i (sources contiguous along i); KI = false: layout [i][k]
// (pitch 36), vectorised along k.  Thread -> element mapping (vid = it*256 + tid):
//   KI : i = 4 * (vid % (TI/4)), k = vid / (TI/4)          !KI : k = 4 * (vid % 8), i = vid / 8
template <int TI>
struct RegTile {
    static constexpr int NV = TI * BK / 4 / NTHR;
    float4 v[NV];
};

template <typename T> __device__ __forceinline__ float ld1(const T* p) { return to_f32<T>(__ldg(p)); }

// p: element (i = 0, k = 0) of this k-tile; si / sk element strides; ni / nk valid extents (elements
// outside read as 0); vec: T is float, the vector dimension has stride 1 and every vector is 16-byte aligned.
template <int TI, bool KI, typename T>
__device__ __forceinline__ void load_raw(RegTile<TI>& r, const T* p, int64_t si, int64_t sk, int ni, int nk, bool vec) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int it = 0; it < RegTile<TI>::NV; ++it) {
        const int vid = it * NTHR + tid;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (KI) {
            const int i = (vid % (TI / 4)) * 4, k = vid / (TI / 4);
            if (k < nk && i < ni) {
                const T* q = p + (int64_t)i * si + (int64_t)k * sk;
                if (sizeof(T) == 4 && vec && i + 3 < ni) {
                    v = __ldg(reinterpret_cast<const float4*>(q));
                } else {
                    v.x = ld1(q);
                    if (i + 1 < ni) v.y = ld1(q + si);
                    if (i + 2 < ni) v.z = ld1(q + 2 * si);
                    if (i + 3 < ni) v.w = ld1(q + 3 * si);
                }
            }
        } else {
            const int k = (vid % (BK / 4)) * 4, i = vid / (BK / 4);
            if (i < ni && k < nk) {
                const T* q = p + (int64_t)i * si + (int64_t)k * sk;
                if (sizeof(T) == 4 && vec && k + 3 < nk) {
                    v = __ldg(reinterpret_cast<const float4*>(q));
                } else {
                    v.x = ld1(q);
                    if (k + 1 < nk) v.y = ld1(q + sk);
                    if (k + 2 < nk) v.z = ld1(q + 2 * sk);
                    if (k + 3 < nk) v.w = ld1(q + 3 * sk);
                }
            }
        }
        r.v[it] = v;
    }
}

// xf(i, k, raw) -> the operand element (decay / dt' factors, causal mask); i, k local to the tile
template <int TI, bool KI, class XF>
__device__ __forceinline__ void store_tile(float* s, const RegTile<TI>& r, XF xf) {
    constexpr int LD = KI ? TI + 8 : BK + 4;
    const int tid = threadIdx.x;
#pragma unroll
    for (int it = 0; it < RegTile<TI>::NV; ++it) {
        const int vid = it * NTHR + tid;
        const float4 v = r.v[it];
        if (KI) {
            const int i = (vid % (TI / 4)) * 4, k = vid / (TI / 4);
            *reinterpret_cast<float4*>(s + k * LD + i) = make_float4(xf(i, k, v.x), xf(i + 1, k, v.y), xf(i + 2, k, v.z), xf(i + 3, k, v.w));
        } else {
            const int k = (vid % (BK / 4)) * 4, i = vid / (BK / 4);
            *reinterpret_cast<float4*>(s + i * LD + k) = make_float4(xf(i, k, v.x), xf(i, k + 1, v.y), xf(i, k + 2, v.z), xf(i, k + 3, v.w));
        }
    }
}

struct Identity {
    __device__ __forceinline__ float operator()(int, int, float v) const { return v; }
};

// can a [rows][cols] float source with these strides be read with aligned 128-bit loads along `vec_stride`'s dimension?
template <typename T>
__device__ __forceinline__ bool vec_ok(const T* p, int64_t vec_stride, int64_t other_stride) {
    return sizeof(T) == 4 && vec_stride == 1 && (other_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0;
}

// Element-wise tile fill used by the backward kernels (not yet on the register-staged pipeline above):
// same layouts; `i_fast` picks the thread -> element mapping so that global reads coalesce along whichever
// of i / k has stride 1 in memory.  f(i, k) returns the (already transformed, bounds-checked) element.
template <int TI, bool KI, class F>
__device__ __forceinline__ void fill_tile(float* s, bool i_fast, F f) {
    constexpr int LD = KI ? TI + 8 : BK + 4;
    const int tid = threadIdx.x;
    if (i_fast) {
#pragma unroll
        for (int it = 0; it < TI * BK / NTHR; ++it) {
            const int idx = it * NTHR + tid;
            const int i = idx % TI, k = idx / TI;
            s[KI ? k * LD + i : i * LD + k] = f(i, k);
        }
    } else {
#pragma unroll
        for (int it = 0; it < TI * BK / NTHR; ++it) {
            const int idx = it * NTHR + tid;
            const int k = idx % BK, i = idx / BK;
            s[KI ? k * LD + i : i * LD + k] = f(i, k);
        }
    }
}

// acc += A_tile (128 x 32) * B_tile (64 x 32)^T for this warp's 32x32 sub-tile.
template <bool A_KM, bool B_KN>
__device__ __forceinline__ void warp_mma(Acc& acc, const float* As, const float* Bs, bool x3) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int m0 = (warp & 3) * 32, n0 = (warp >> 2) * 32;
#pragma unroll
    for (int ks = 0; ks < BK / 8; ++ks) {
        const int k0 = ks * 8;
        uint32_t ah[2][4], al[2][4], bh[4][2], bl[4][2];
#pragma unroll
        for (int mi = 0; mi < 2; ++mi) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int m = m0 + mi * 16 + g + ((r & 1) ? 8 : 0);
                const int k = k0 + t + ((r & 2) ? 4 : 0);
                const float a = As[A_KM ? k * LDA_KM + m : m * LDA_MK + k];
                ah[mi][r] = tf32_rna(a);
                al[mi][r] = tf32_rna(a - __uint_as_float(ah[mi][r]));
            }
        }
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int n = n0 + ni * 8 + g;
                const int k = k0 + t + (r ? 4 : 0);
                const float b = Bs[B_KN ? k * LDB_KN + n : n * LDB_NK + k];
                bh[ni][r] = tf32_rna(b);
                bl[ni][r] = tf32_rna(b - __uint_as_float(bh[ni][r]));
            }
        }
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) {
                if (x3) {  // small terms first
                    mma_tf32(acc.v[mi][ni], al[mi], bh[ni]);
                    mma_tf32(acc.v[mi][ni], ah[mi], bl[ni]);
                }
                mma_tf32(acc.v[mi][ni], ah[mi], bh[ni]);
            }
    }
}

// visit every accumulator element of this thread: fn(m, n, value&) with m in [0,128), n in [0,64)
template <class F>
__device__ __forceinline__ void for_each_acc(Acc& acc, F fn) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int m0 = (warp & 3) * 32, n0 = (warp >> 2) * 32;
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int r = 0; r < 4; ++r) fn(m0 + mi * 16 + g + ((r & 2) ? 8 : 0), n0 + ni * 8 + 2 * t + (r & 1), acc.v[mi][ni][r]);
}

struct Smem {
    float A[2][A_FLOATS];
    float B[2][B_FLOATS];
    float cs[2][MAXQ];
    float dtp[2][MAXQ];
    float v1[2][MAXQ];            // per-position factor vectors (kernel specific)
    float v2[2][MAXQ];
    float rowf[MAXQ / BK][BM];    // per (k-tile, row) decay factors of the diagonal-block contractions
    float red[8];
    int sid[MAXQ];                // seq_idx of the chunk's positions (SEQ instantiations)
};

// One software-pipelined pass over nkt k-tiles: the raw tile kt+1 is fetched into registers while the
// tensor cores work on tile kt; la/lb(kt, regs) load, sa/sb(kt, regs, smem) transform + store, mm(A, B) multiplies.
// Ends with a barrier, so the caller may start another pass (or re-use shared memory) right away.
template <class LA, class LB, class SA, class SB, class MM>
__device__ __forceinline__ void gemm_pipeline(Smem& sm, int nkt, LA la, LB lb, SA sa, SB sb, MM mm) {
    if (nkt <= 0) return;
    RegTile<BM> ra;
    RegTile<BN> rb;
    la(0, ra);
    lb(0, rb);
    sa(0, ra, sm.A[0]);
    sb(0, rb, sm.B[0]);
    __syncthreads();
    for (int kt = 0; kt < nkt; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nkt) {
            la(kt + 1, ra);
            lb(kt + 1, rb);
        }
        mm(sm.A[buf], sm.B[buf]);
        if (kt + 1 < nkt) {
            sa(kt + 1, ra, sm.A[buf ^ 1]);
            sb(kt + 1, rb, sm.B[buf ^ 1]);
        }
        __syncthreads();
    }
}

// ---- engine A: warp-level mma.sync tiles (accumulators in registers) ---------------------------------------
struct MmaEngine {
    using Shared = Smem;
    static constexpr int MIN_CTAS = 2;   // accumulators in registers: 128 registers per thread
    Acc acc;
    static __device__ __forceinline__ Shared& smem() {
        extern __shared__ __align__(1024) unsigned char raw[];
        return *reinterpret_cast<Shared*>(raw);
    }
    template <int TI, bool KI, typename T>
    static __device__ __forceinline__ void load(RegTile<TI>& r, const T* p, int64_t si, int64_t sk, int ni, int nk, bool vec) {
        load_raw<TI, KI>(r, p, si, sk, ni, nk, vec);
    }
    template <int TI, bool KI, class XF>
    static __device__ __forceinline__ void store(float* s, const RegTile<TI>& r, XF xf) { store_tile<TI, KI>(s, r, xf); }
    __device__ __forceinline__ void begin(Shared&) { acc.zero(); }
    template <bool KIA, bool KIB, class LA, class LB, class SA, class SB>
    __device__ __forceinline__ void pass(Shared& sm, int nkt, bool x3, LA la, LB lb, SA sa, SB sb) {
        gemm_pipeline(sm, nkt, la, lb, sa, sb, [&](const float* sA, const float* sB) { warp_mma<KIA, KIB>(acc, sA, sB, x3); });
    }
    template <class F> __device__ __forceinline__ void for_each(Shared&, F fn) { for_each_acc(acc, fn); }
    __device__ __forceinline__ void end(Shared&) {}
};

// ---- engine B: tcgen05 (UMMA) tiles: operands in the canonical no-swizzle K-major shared-memory layout, fp32
//      accumulators in tensor memory, one thread issues the MMAs, completion through mbarriers -------------------
// byte offset of operand element (row i, k) inside a [TI rows x 32 k] tile:
//     (k / 4) * LBO + (i / 8) * SBO + (i % 8) * 16 + (k % 4) * 4
// i.e. 8-row x 16-byte core matrices (cute/atom/mma_traits_sm100.hpp, "LayoutType::INTERLEAVE ((8,n),2):((1,SBO),LBO)").
// SBO and LBO are free descriptor fields: padding them (144 instead of 128, +16) makes both store patterns below
// bank-conflict free -- a quarter warp storing the eight 16-byte k-chunks of one row, and a warp storing single
// words of 8 row-quads x 4 consecutive k.  Validated bit-exactly by tools/tc_probe.cu.
namespace tc {
constexpr int SBO = 144;
template <int TI> struct Geo {
    static constexpr int LBO = (TI / 8) * SBO + 16;
    static constexpr int BYTES = (BK / 4) * LBO;
};
constexpr int A_BYTES = Geo<BM>::BYTES, B_BYTES = Geo<BN>::BYTES;   // 18560, 9344
constexpr int TMEM_COLS = BN;                                        // 128 lanes x 64 fp32 columns

struct Shared {
    float cs[2][MAXQ];
    float dtp[2][MAXQ];
    float v1[2][MAXQ];
    float v2[2][MAXQ];
    float rowf[MAXQ / BK][BM];
    float red[8];
    int sid[MAXQ];
    uint64_t bar[2];      // "the MMAs that read operand stage s have completed"
    uint64_t bar_done;
    uint32_t tmem_slot, pad_;
    alignas(128) unsigned char Ahi[2][A_BYTES];
    alignas(128) unsigned char Bhi[2][B_BYTES];
    alignas(128) unsigned char Alo[2][A_BYTES];   // low parts of the 3xTF32 split (allocated only in that mode)
    alignas(128) unsigned char Blo[2][B_BYTES];
};
constexpr size_t SMEM_TF32 = offsetof(Shared, Alo), SMEM_X3 = sizeof(Shared);

struct Dst {   // where one operand stage goes
    unsigned char* hi;
    unsigned char* lo;
    bool x3;
};

__device__ __forceinline__ unsigned s32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(unsigned saddr, unsigned lbo, unsigned sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46);   // version 1 (Blackwell), no swizzle, base offset 0
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}" ::"r"(
            s32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n}" ::"r"(tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
}  // namespace tc

#ifndef B200_SSD_TC_CTAS
#define B200_SSD_TC_CTAS 2
#endif
struct TcEngine {
    using Shared = tc::Shared;
    // resident CTAs per SM.  Measured at the MedSSD stage-0 shape, TF32 mode (fwd / bwd of one call): 1 CTA 5.06 / 14.3 ms,
    // 2 CTAs 3.90 / 10.9 ms, 3 CTAs (80 registers, no spills, 66 KB of shared memory each) 4.27 / 11.7 ms -- beyond two the
    // staging stores saturate the shared-memory pipe (56-65 % of its wavefront peak at two CTAs) instead of hiding more latency
    static constexpr int MIN_CTAS = B200_SSD_TC_CTAS;
    uint32_t tmem;
    uint32_t issued[2], waited[2];
    bool started, x3_;
    static __device__ __forceinline__ Shared& smem() {
        extern __shared__ __align__(1024) unsigned char raw[];
        return *reinterpret_cast<Shared*>(raw);
    }
    // register-tile mappings.  !KI: as load_raw (vid = it * 256 + tid: k = 4 (vid % 8), i = vid / 8).
    // KI (the source is contiguous along i): a thread owns a block of 4 rows x NV consecutive k -- row quad iq = tid % (TI/4),
    // k = NV (tid / (TI/4)) + it -- so its NV 128-bit loads (one per k, lanes of a warp along i: 512-byte runs) become 4 stores
    // of NV consecutive k of ONE row each (one STS.128 for the 128-row operand, one STS.64 for the 64-row operand) in the
    // K-major core-matrix layout.  The first version gave a thread 4 rows x 1 k per load and stored single words:
    // 16 STS.32 per k-tile and thread for the 128-row operand instead of 4 STS.128.
    template <int TI> static __device__ __forceinline__ void ki_map(int tid, int& i, int& k0) {
        i = 4 * (tid % (TI / 4));
        k0 = RegTile<TI>::NV * (tid / (TI / 4));
    }
    template <int TI, bool KI, typename T>
    static __device__ __forceinline__ void load(RegTile<TI>& r, const T* p, int64_t si, int64_t sk, int ni, int nk, bool vec) {
        if constexpr (!KI) {
            load_raw<TI, false>(r, p, si, sk, ni, nk, vec);
        } else {
            int i, k0;
            ki_map<TI>(threadIdx.x, i, k0);
#pragma unroll
            for (int it = 0; it < RegTile<TI>::NV; ++it) {
                const int k = k0 + it;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < nk && i < ni) {
                    const T* q = p + (int64_t)i * si + (int64_t)k * sk;
                    if (sizeof(T) == 4 && vec && i + 3 < ni) {
                        v = __ldg(reinterpret_cast<const float4*>(q));
                    } else {
                        v.x = ld1(q);
                        if (i + 1 < ni) v.y = ld1(q + si);
                        if (i + 2 < ni) v.z = ld1(q + 2 * si);
                        if (i + 3 < ni) v.w = ld1(q + 3 * si);
                    }
                }
                r.v[it] = v;
            }
        }
    }
    // run-time choice of the mapping: ki = "i is the contiguous dimension of the source"
    template <int TI, typename T>
    static __device__ __forceinline__ void load_any(RegTile<TI>& r, const T* p, int64_t si, int64_t sk, int ni, int nk, bool ki) {
        if (ki) load<TI, true>(r, p, si, sk, ni, nk, vec_ok(p, si, sk));
        else load<TI, false>(r, p, si, sk, ni, nk, vec_ok(p, sk, si));
    }
    template <int TI, class XF>
    static __device__ __forceinline__ void store_any(const tc::Dst& d, const RegTile<TI>& r, bool ki, XF xf) {
        if (ki) store<TI, true>(d, r, xf);
        else store<TI, false>(d, r, xf);
    }
    static __device__ __forceinline__ float hi_part(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }
    template <int TI, bool KI, class XF>
    static __device__ __forceinline__ void store(const tc::Dst& d, const RegTile<TI>& r, XF xf) {
        constexpr int LBO = tc::Geo<TI>::LBO;
        const int tid = threadIdx.x;
#pragma unroll
        for (int it = 0; it < RegTile<TI>::NV; ++it) {
            const int vid = it * NTHR + tid;
            const float4 v = r.v[it];
            if constexpr (!KI) {
                const int k = (vid % (BK / 4)) * 4, i = vid / (BK / 4);
                const int off = (k >> 2) * LBO + (i >> 3) * tc::SBO + (i & 7) * 16;
                float4 t = make_float4(xf(i, k, v.x), xf(i, k + 1, v.y), xf(i, k + 2, v.z), xf(i, k + 3, v.w));
                if (d.x3) {
                    const float4 h = make_float4(hi_part(t.x), hi_part(t.y), hi_part(t.z), hi_part(t.w));
                    *reinterpret_cast<float4*>(d.lo + off) = make_float4(t.x - h.x, t.y - h.y, t.z - h.z, t.w - h.w);
                    t = h;
                }
                *reinterpret_cast<float4*>(d.hi + off) = t;
            }
        }
        if constexpr (KI) {
            constexpr int NV = RegTile<TI>::NV;   // 4 (128-row operand) or 2 (64-row operand) consecutive k per row
            int i, k0;
            ki_map<TI>(tid, i, k0);
            float t[4][NV];
#pragma unroll
            for (int it = 0; it < NV; ++it) {
                const float4 v = r.v[it];
                t[0][it] = xf(i, k0 + it, v.x);
                t[1][it] = xf(i + 1, k0 + it, v.y);
                t[2][it] = xf(i + 2, k0 + it, v.z);
                t[3][it] = xf(i + 3, k0 + it, v.w);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int off = (k0 >> 2) * LBO + ((i + j) >> 3) * tc::SBO + ((i + j) & 7) * 16 + (k0 & 3) * 4;
                float h[NV];
#pragma unroll
                for (int it = 0; it < NV; ++it) h[it] = t[j][it];
                if (d.x3) {
                    float lo[NV];
#pragma unroll
                    for (int it = 0; it < NV; ++it) {
                        h[it] = hi_part(t[j][it]);
                        lo[it] = t[j][it] - h[it];
                    }
                    if constexpr (NV == 4) *reinterpret_cast<float4*>(d.lo + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                    else *reinterpret_cast<float2*>(d.lo + off) = make_float2(lo[0], lo[1]);
                }
                if constexpr (NV == 4) *reinterpret_cast<float4*>(d.hi + off) = make_float4(h[0], h[1], h[2], h[3]);
                else *reinterpret_cast<float2*>(d.hi + off) = make_float2(h[0], h[1]);
            }
        }
    }
    // call after every early-return of the CTA: allocates tensor memory, arms the barriers (contains a block barrier)
    __device__ __forceinline__ void begin(Shared& sm) {
        if (threadIdx.x < 32) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::s32(&sm.tmem_slot)), "r"(tc::TMEM_COLS));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
        }
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc::s32(&sm.bar[0])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc::s32(&sm.bar[1])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc::s32(&sm.bar_done)) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem = sm.tmem_slot;
        issued[0] = issued[1] = waited[0] = waited[1] = 0;
        started = false;
    }
    template <bool KIA, bool KIB, class LA, class LB, class SA, class SB>
    __device__ __forceinline__ void pass(Shared& sm, int nkt, bool x3, LA la, LB lb, SA sa, SB sb) {
        if (nkt <= 0) return;
        x3_ = x3;
        RegTile<BM> ra;
        RegTile<BN> rb;
        la(0, ra);
        lb(0, rb);
        // D = F32, A = B = TF32, both K-major, M = 128, N = 64
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        for (int kt = 0; kt < nkt; ++kt) {
            const int buf = kt & 1;
            if (issued[buf] > waited[buf]) {   // the MMAs that read this stage two tiles ago must be done
                tc::mbar_wait(&sm.bar[buf], waited[buf] & 1);
                ++waited[buf];
            }
            sa(kt, ra, tc::Dst{sm.Ahi[buf], sm.Alo[buf], x3});
            sb(kt, rb, tc::Dst{sm.Bhi[buf], sm.Blo[buf], x3});
            if (kt + 1 < nkt) {   // next tile's global loads fly while the tensor core works
                la(kt + 1, ra);
                lb(kt + 1, rb);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the MMA
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            if (threadIdx.x == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const unsigned ah = tc::s32(sm.Ahi[buf]), bh = tc::s32(sm.Bhi[buf]), al = tc::s32(sm.Alo[buf]), bl = tc::s32(sm.Blo[buf]);
                constexpr unsigned LA_ = tc::Geo<BM>::LBO, LB_ = tc::Geo<BN>::LBO;
#pragma unroll
                for (int ks = 0; ks < BK / 8; ++ks) {   // one MMA = 8 TF32 along K = two 16-byte core columns
                    const unsigned oa = ks * 2 * LA_, ob = ks * 2 * LB_;
                    if (x3) {   // small terms first
                        tc::umma_tf32(tmem, tc::make_desc(al + oa, LA_, tc::SBO), tc::make_desc(bh + ob, LB_, tc::SBO), idesc, started);
                        tc::umma_tf32(tmem, tc::make_desc(ah + oa, LA_, tc::SBO), tc::make_desc(bl + ob, LB_, tc::SBO), idesc, 1u);
                        tc::umma_tf32(tmem, tc::make_desc(ah + oa, LA_, tc::SBO), tc::make_desc(bh + ob, LB_, tc::SBO), idesc, 1u);
                    } else {
                        tc::umma_tf32(tmem, tc::make_desc(ah + oa, LA_, tc::SBO), tc::make_desc(bh + ob, LB_, tc::SBO), idesc, started);
                    }
                    started = true;
                }
                tc::umma_commit(&sm.bar[buf]);
            }
            started = true;
            ++issued[buf];
        }
    }
    // visit every accumulator element: fn(m, n, value&) -- thread = one row (TMEM lane), 32 consecutive columns
    template <class F> __device__ __forceinline__ void for_each(Shared& sm, F fn) {
        if (threadIdx.x == 0) tc::umma_commit(&sm.bar_done);
        tc::mbar_wait(&sm.bar_done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const int m = (warp & 3) * 32 + lane, n0 = (warp >> 2) * 32;
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 8) {
            uint32_t v[8];
            const uint32_t addr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(n0 + c0);
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                         : "r"(addr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float f = started ? __uint_as_float(v[j]) : 0.f;
                fn(m, n0 + c0 + j, f);
            }
        }
    }
    __device__ __forceinline__ void end(Shared& sm) {
        (void)sm;
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tc::TMEM_COLS));
    }
};

__device__ __forceinline__ Smem& smem_ref() {
    extern __shared__ __align__(1024) unsigned char raw[];
    return *reinterpret_cast<Smem*>(raw);
}

// stage the (b, h, c) chunk's cs / dt' rows into shared memory buffer `hb`
template <class S>
__device__ __forceinline__ void stage_cs(S& sm, int hb, const Ws& ws, const Dims& d, int b, int h, int c) {
    const size_t off = (((size_t)b * d.H + h) * d.nc + c) * d.Q;
    for (int i = threadIdx.x; i < d.Q; i += NTHR) {
        sm.cs[hb][i] = ws.cs[off + i];
        sm.dtp[hb][i] = ws.dtp[off + i];
    }
}

// stage chunk c's seq_idx values into shared memory (no barrier)
template <class S>
__device__ __forceinline__ void stage_sid(S& sm, const Dims& d, int b, int c) {
    for (int i = threadIdx.x; i < d.Q; i += NTHR) sm.sid[i] = seq_at(d, b, c, i);
}

template <class S>
__device__ __forceinline__ float block_sum(S& sm, float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < NTHR / 32; ++w) s += sm.red[w];
    return s;
}

// ---- K1: dt' = clamp(softplus(dt + bias)), cs = inclusive cumsum(dt' A) within each chunk -----
template <typename T>
__global__ void __launch_bounds__(MAXQ) dt_cumsum_kernel(const T* dt, int64_t s0, int64_t s1, int64_t s2, const float* A,
                                                         const float* dt_bias, int softplus, float dt_min, float dt_max, Dims d,
                                                         Ws ws) {
    __shared__ float wsum[MAXQ / 32];
    const int c = blockIdx.x % d.nc, h = (blockIdx.x / d.nc) % d.H, b = blockIdx.x / (d.nc * d.H);
    const int i = threadIdx.x, l = c * d.Q + i;
    float v = 0.f;
    if (i < d.Q && l < d.L) {
        v = to_f32<T>(__ldg(dt + b * s0 + l * s1 + h * s2)) + (dt_bias ? __ldg(dt_bias + h) : 0.f);
        if (softplus) v = softplus20(v);
        v = fminf(fmaxf(v, dt_min), dt_max);
    }
    float x = v * __ldg(A + h);
    const int lane = i & 31, w = i >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    float pre = 0.f;
    for (int j = 0; j < w; ++j) pre += wsum[j];
    x += pre;
    if (i < d.Q) {
        const size_t off = (((size_t)b * d.H + h) * d.nc + c) * d.Q + i;
        ws.dtp[off] = v;
        ws.cs[off] = x;
    }
}

// ---- K2 / B1: per (b, c, h):  out[p][n] = sum_s w_s src_x[s, p] src_b[s, n] -----------------------
//   MODE 0 (chunk states):  src_x = x,    src_b = B,  w_s = exp(cs_Q - cs_s) dt'_s
//   MODE 1 (d states):      src_x = dout, src_b = C,  w_s = exp(cs_s)
// GEMM: M = n (128 per tile), N = p (64 per tile), K = s.
template <typename T, int MODE, class E, bool SEQ>
__global__ void __launch_bounds__(NTHR, E::MIN_CTAS) chunk_state_kernel(View4<T> X, View4<T> Bv, Dims d, Ws ws, float* out, int x3) {
    typename E::Shared& sm = E::smem();
    const int ntn = (d.N + BM - 1) / BM, ntp = (d.P + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tn = bid % ntn; bid /= ntn;
    const int tp = bid % ntp; bid /= ntp;
    const int h = bid % d.H; bid /= d.H;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int g = h / d.hpg;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int n0 = tn * BM, p0 = tp * BN;
    stage_cs(sm, 0, ws, d, b, h, c);
    __syncthreads();
    const float csQ = sm.cs[0][d.Q - 1];
    for (int i = threadIdx.x; i < d.Q; i += NTHR)
        sm.v1[0][i] = MODE == 0 ? exp_acc(csQ - sm.cs[0][i]) * sm.dtp[0][i] : exp_acc(sm.cs[0][i]);
    if (SEQ) {   // MODE 0: only the sequence still open at the chunk's end; MODE 1: only the one entering the chunk
        const int ref = MODE == 0 ? seq_end(d, b, c) : seq_prev(d, b, c);
        for (int i = threadIdx.x; i < d.Q; i += NTHR)
            if (seq_at(d, b, c, i) != ref) sm.v1[0][i] = 0.f;
    }
    __syncthreads();
    const T* pa = Bv.p + b * Bv.s0 + (int64_t)l0 * Bv.s1 + g * Bv.s2 + (int64_t)n0 * Bv.s3;   // (i = n, k = s)
    const T* pb = X.p + b * X.s0 + (int64_t)l0 * X.s1 + h * X.s2 + (int64_t)p0 * X.s3;        // (i = p, k = s)
    const bool va = vec_ok(pa, Bv.s1, Bv.s3), vb = vec_ok(pb, X.s1, X.s3);
    E eng;
    eng.begin(sm);
    eng.template pass<false, false>(
        sm, (q + BK - 1) / BK, x3 != 0,
        [&](int kt, RegTile<BM>& r) { E::template load<BM, false>(r, pa + (int64_t)kt * BK * Bv.s1, Bv.s3, Bv.s1, d.N - n0, q - kt * BK, va); },
        [&](int kt, RegTile<BN>& r) { E::template load<BN, false>(r, pb + (int64_t)kt * BK * X.s1, X.s3, X.s1, d.P - p0, q - kt * BK, vb); },
        [&](int, const RegTile<BM>& r, auto sA) { E::template store<BM, false>(sA, r, Identity()); },
        [&](int kt, const RegTile<BN>& r, auto sB) {
            const float* w = sm.v1[0] + kt * BK;
            E::template store<BN, false>(sB, r, [&](int, int k, float v) { return v * w[k]; });
        });
    float* o = out + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N;
    eng.for_each(sm, [&](int m, int n, float& v) {
        const int nn = n0 + m, p = p0 + n;
        if (nn < d.N && p < d.P) o[(size_t)p * d.N + nn] = v;
    });
    eng.end(sm);
}

// ---- K3: state passing over chunks (in place: local states -> chunk-entry states) --------------
// HBM-bound streaming pass: 128-bit accesses, 32-bit indexing, and the loads of 8 chunks are issued before the
// (sequential) recurrence over them so each thread keeps 8 independent 16-byte requests in flight.
constexpr int SPB = 8;  // chunks per batch of loads
template <bool SEQ>
__global__ void __launch_bounds__(256) state_pass_kernel(Dims d, Ws ws, const float* init, float* fin) {
    const int PN4 = d.P * d.N / 4;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= PN4) return;
    const int h = blockIdx.y % d.H, b = blockIdx.y / d.H;
    const size_t cstride = (size_t)d.H * PN4;                                       // float4 units between chunks
    float4* st = reinterpret_cast<float4*>(ws.states) + ((size_t)b * d.nc * d.H + h) * PN4 + e;
    const float* csq = ws.cs + ((size_t)b * d.H + h) * d.nc * d.Q + d.Q - 1;
    float4 run = init ? reinterpret_cast<const float4*>(init)[((size_t)b * d.H + h) * PN4 + e] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c0 = 0; c0 < d.nc; c0 += SPB) {
        float4 loc[SPB];
        float dec[SPB];
#pragma unroll
        for (int k = 0; k < SPB; ++k)
            if (c0 + k < d.nc) {
                loc[k] = st[(size_t)(c0 + k) * cstride];
                dec[k] = exp_acc(__ldg(csq + (size_t)(c0 + k) * d.Q));
                if (SEQ && seq_end(d, b, c0 + k) != seq_prev(d, b, c0 + k)) dec[k] = 0.f;   // a sequence starts in the chunk
            }
#pragma unroll
        for (int k = 0; k < SPB; ++k)
            if (c0 + k < d.nc) {
                st[(size_t)(c0 + k) * cstride] = run;
                run = make_float4(fmaf(dec[k], run.x, loc[k].x), fmaf(dec[k], run.y, loc[k].y), fmaf(dec[k], run.z, loc[k].z),
                                  fmaf(dec[k], run.w, loc[k].w));
            }
    }
    if (fin) reinterpret_cast<float4*>(fin)[((size_t)b * d.H + h) * PN4 + e] = run;
}
// element-wise fallback (P * N not a multiple of 4)
template <bool SEQ>
__global__ void state_pass_kernel_scalar(Dims d, Ws ws, const float* init, float* fin) {
    const size_t PN = (size_t)d.P * d.N;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)d.batch * d.H * PN) return;
    const size_t e = idx % PN;
    const int h = (idx / PN) % d.H, b = idx / (PN * d.H);
    float run = init ? init[idx] : 0.f;
    for (int c = 0; c < d.nc; ++c) {
        float* s = ws.states + (((size_t)b * d.nc + c) * d.H + h) * PN + e;
        const float loc = *s;
        *s = run;
        const float csQ = ws.cs[(((size_t)b * d.H + h) * d.nc + c) * d.Q + d.Q - 1];
        const float dec = (SEQ && seq_end(d, b, c) != seq_prev(d, b, c)) ? 0.f : exp_acc(csQ);
        run = dec * run + loc;
    }
    if (fin) fin[idx] = run;
}

// ---- K4: CB[l][s] = sum_n C[l, n] B[s, n]  per (b, c, g); only tiles touching s <= l ------------
template <typename T, class E>
__global__ void __launch_bounds__(NTHR, E::MIN_CTAS) cb_kernel(View4<T> Cv, View4<T> Bv, Dims d, Ws ws, int x3) {
    typename E::Shared& sm = E::smem();
    const int ntm = (d.Q + BM - 1) / BM, ntn = (d.Q + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tn = bid % ntn; bid /= ntn;
    const int tm = bid % ntm; bid /= ntm;
    const int g = bid % d.G; bid /= d.G;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, s0 = tn * BN;
    if (m0 >= q || s0 >= q || s0 > m0 + BM - 1) return;
    const T* pa = Cv.p + b * Cv.s0 + (int64_t)(l0 + m0) * Cv.s1 + g * Cv.s2;   // (i = l, k = n)
    const T* pb = Bv.p + b * Bv.s0 + (int64_t)(l0 + s0) * Bv.s1 + g * Bv.s2;   // (i = s, k = n)
    const bool va = vec_ok(pa, Cv.s1, Cv.s3), vb = vec_ok(pb, Bv.s1, Bv.s3);
    E eng;
    eng.begin(sm);
    eng.template pass<true, true>(
        sm, (d.N + BK - 1) / BK, x3 != 0,
        [&](int kt, RegTile<BM>& r) { E::template load<BM, true>(r, pa + (int64_t)kt * BK * Cv.s3, Cv.s1, Cv.s3, q - m0, d.N - kt * BK, va); },
        [&](int kt, RegTile<BN>& r) { E::template load<BN, true>(r, pb + (int64_t)kt * BK * Bv.s3, Bv.s1, Bv.s3, q - s0, d.N - kt * BK, vb); },
        [&](int, const RegTile<BM>& r, auto sA) { E::template store<BM, true>(sA, r, Identity()); },
        [&](int, const RegTile<BN>& r, auto sB) { E::template store<BN, true>(sB, r, Identity()); });
    float* o = ws.cb + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    eng.for_each(sm, [&](int m, int n, float& v) {
        const int l = m0 + m, s = s0 + n;
        if (l < q && s < q) o[(size_t)l * d.Q + s] = v;
    });
    eng.end(sm);
}

// ---- K5: y = (CB o decay) (dt' x) + exp(cs) C Sin^T + D x   per (b, c, h) ------------------------
// decay(l, s) = exp(cs_l - cs_s) is applied to the CB tile on its way into shared memory.  For rows below the
// 32-wide k-tile it is the product of two factors <= 1 (reference point: cs at the end of the k-tile), one
// per row and one per column, precomputed once per CTA; inside the 32 x 32 diagonal block it is evaluated
// exactly per element (no overflow whatever the decay rate).
template <typename T, class E, bool SEQ>
__global__ void __launch_bounds__(NTHR, E::MIN_CTAS) chunk_scan_kernel(View4<T> X, View4<T> Cv, const float* D, Dims d, Ws ws, T* out,
                                                             int64_t o0, int64_t o1, int64_t o2, int64_t o3, int has_init, int x3) {
    typename E::Shared& sm = E::smem();
    const int ntm = (d.Q + BM - 1) / BM, ntp = (d.P + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tp = bid % ntp; bid /= ntp;
    const int tm = bid % ntm; bid /= ntm;
    const int h = bid % d.H; bid /= d.H;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int g = h / d.hpg;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, p0 = tp * BN;
    if (m0 >= q) return;
    stage_cs(sm, 0, ws, d, b, h, c);
    if (SEQ) stage_sid(sm, d, b, c);
    __syncthreads();
    const int send = min(q, m0 + BM), nkt1 = (send + BK - 1) / BK;
    const int sprev = SEQ ? seq_prev(d, b, c) : 0;
    for (int i = threadIdx.x; i < d.Q; i += NTHR) {
        const float ref = sm.cs[0][min((i / BK) * BK + BK - 1, d.Q - 1)];
        sm.v1[0][i] = exp_acc(ref - sm.cs[0][i]) * sm.dtp[0][i];   // column factor (<= dt')
        sm.v2[0][i] = exp_acc(sm.cs[0][i]);                        // exp(cs_l) of the state term
        if (SEQ && sm.sid[i] != sprev) sm.v2[0][i] = 0.f;          // the chunk-entry state belongs to another sequence
    }
    for (int idx = threadIdx.x; idx < nkt1 * BM; idx += NTHR) {
        const int kt = idx / BM, i = idx % BM;
        const float ref = sm.cs[0][min(kt * BK + BK - 1, d.Q - 1)];
        sm.rowf[kt][i] = exp_acc(sm.cs[0][min(m0 + i, d.Q - 1)] - ref);   // used for rows below the k-tile only (<= 1)
    }
    __syncthreads();
    const float* cb = ws.cb + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q + (size_t)m0 * d.Q;   // (i = l, k = s)
    const T* px = X.p + b * X.s0 + (int64_t)l0 * X.s1 + h * X.s2 + (int64_t)p0 * X.s3;                      // (i = p, k = s)
    const bool va = vec_ok(cb, 1, d.Q), vb = vec_ok(px, X.s1, X.s3);
    E eng;
    eng.begin(sm);
    eng.template pass<false, false>(
        sm, nkt1, x3 != 0,
        [&](int kt, RegTile<BM>& r) { E::template load<BM, false>(r, cb + kt * BK, d.Q, 1, q - m0, send - kt * BK, va); },
        [&](int kt, RegTile<BN>& r) { E::template load<BN, false>(r, px + (int64_t)kt * BK * X.s1, X.s3, X.s1, d.P - p0, q - kt * BK, vb); },
        [&](int kt, const RegTile<BM>& r, auto sA) {
            const int k0 = kt * BK;
            E::template store<BM, false>(sA, r, [&](int i, int k, float v) {
                const int l = m0 + i, s = k0 + k;
                if (s > l) return 0.f;
                if (SEQ && sm.sid[min(l, d.Q - 1)] != sm.sid[s]) return 0.f;
                if (l < k0 + BK) return v * exp_acc(sm.cs[0][l] - sm.cs[0][s]) * sm.dtp[0][s];
                return v * sm.rowf[kt][i] * sm.v1[0][s];
            });
        },
        [&](int, const RegTile<BN>& r, auto sB) { E::template store<BN, false>(sB, r, Identity()); });
    if (c > 0 || has_init) {  // contribution of the chunk-entry state (identically zero for the first chunk without initial_states)
        const T* pc = Cv.p + b * Cv.s0 + (int64_t)(l0 + m0) * Cv.s1 + g * Cv.s2;                                   // (i = l, k = n)
        const float* Sin = ws.states + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N + (size_t)p0 * d.N;   // (i = p, k = n)
        const bool vc = vec_ok(pc, Cv.s1, Cv.s3), vs = vec_ok(Sin, 1, d.N);
        eng.template pass<true, false>(
        sm, (d.N + BK - 1) / BK, x3 != 0,
            [&](int kt, RegTile<BM>& r) { E::template load<BM, true>(r, pc + (int64_t)kt * BK * Cv.s3, Cv.s1, Cv.s3, q - m0, d.N - kt * BK, vc); },
            [&](int kt, RegTile<BN>& r) { E::template load<BN, false>(r, Sin + kt * BK, d.N, 1, d.P - p0, d.N - kt * BK, vs); },
            [&](int, const RegTile<BM>& r, auto sA) {
                E::template store<BM, true>(sA, r, [&](int i, int, float v) { return v * sm.v2[0][min(m0 + i, d.Q - 1)]; });
            },
            [&](int, const RegTile<BN>& r, auto sB) { E::template store<BN, false>(sB, r, Identity()); });
    }
    const float Dh = D ? __ldg(D + h) : 0.f;
    eng.for_each(sm, [&](int m, int n, float& v) {
        const int l = m0 + m, p = p0 + n;
        if (l < q && p < d.P) {
            const float y = v + Dh * X.at(b, l0 + l, h, p);
            out[b * o0 + (l0 + l) * o1 + h * o2 + p * o3] = from_f32<T>(y);
        }
    });
    eng.end(sm);
}

// ---- B2: reverse state passing: dstates[c] (off-diagonal adjoint) -> G[c] = adjoint of Sin[c+1];
//          dcsQ[b][h][c] = <G[c], Sin[c+1]>  (accumulated with atomics; caller zero-fills) ----------
// Same streaming structure as K3 (128-bit, 8 chunks of loads in flight); the per-chunk dot products are kept in
// registers and block-reduced once per batch of chunks.
// State gradients (each NULL unless the caller asks): dfin seeds G[nc-1] (otherwise zero, and its dcsQ term, whose
// Sin[nc] is the forward's final states fin, is skipped); dinit receives the adjoint of Sin[0] left after chunk 0.
// With seq_idx the existing masks confine both: dec[0] = 0 when a sequence starts in chunk 0, and B1 keeps only
// the positions of id 0 in chunk 0's off-diagonal adjoint.
template <bool SEQ>
__global__ void __launch_bounds__(NTHR) state_pass_bwd_kernel(Dims d, Ws ws, float* dstates, float* dcsQ, const float* fin,
                                                              const float* dfin, float* dinit) {
    __shared__ float red[NTHR / 32][SPB];
    const int PN4 = d.P * d.N / 4;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = e < PN4;
    const int h = blockIdx.y % d.H, b = blockIdx.y / d.H;
    const size_t cstride = (size_t)d.H * PN4;
    float4* ds = reinterpret_cast<float4*>(dstates) + ((size_t)b * d.nc * d.H + h) * PN4 + (ok ? e : 0);
    const float4* sn = reinterpret_cast<const float4*>(ws.states) + ((size_t)b * d.nc * d.H + h) * PN4 + (ok ? e : 0);
    const float* csq = ws.cs + ((size_t)b * d.H + h) * d.nc * d.Q + d.Q - 1;
    float* dq = dcsQ + ((size_t)b * d.H + h) * d.nc;
    const size_t bh4 = ((size_t)b * d.H + h) * PN4 + (ok ? e : 0);   // this thread's float4 of a (batch, H, P, N) tensor
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 run = z4;
    if (dfin) {   // G[nc-1] = dfin and its term dcsQ[nc-1] = <dfin, fin>, before the loop so that the loop keeps its registers
        float dot = 0.f;
        if (ok) {
            run = reinterpret_cast<const float4*>(dfin)[bh4];
            const float4 f = reinterpret_cast<const float4*>(fin)[bh4];
            dot = run.x * f.x + run.y * f.y + run.z * f.z + run.w * f.w;
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][0] = dot;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < NTHR / 32; ++w) t += red[w][0];
            atomicAdd(dq + d.nc - 1, t);
        }
        __syncthreads();
    }
    for (int c0 = d.nc - 1; c0 >= 0; c0 -= SPB) {   // chunks c0, c0-1, ...
        float4 off[SPB], nxt[SPB];
        float dec[SPB], dot[SPB];
#pragma unroll
        for (int k = 0; k < SPB; ++k) {
            const int c = c0 - k;
            off[k] = z4; nxt[k] = z4; dec[k] = 0.f;
            if (c >= 0) {
                if (ok) off[k] = ds[(size_t)c * cstride];
                if (ok && c + 1 < d.nc) nxt[k] = sn[(size_t)(c + 1) * cstride];
                dec[k] = exp_acc(__ldg(csq + (size_t)c * d.Q));
                if (SEQ && seq_end(d, b, c) != seq_prev(d, b, c)) dec[k] = 0.f;   // no adjoint carry across a reset
            }
        }
#pragma unroll
        for (int k = 0; k < SPB; ++k) {
            const int c = c0 - k;
            dot[k] = 0.f;
            if (c >= 0) {
                if (ok) ds[(size_t)c * cstride] = run;
                dot[k] = run.x * nxt[k].x + run.y * nxt[k].y + run.z * nxt[k].z + run.w * nxt[k].w;
                run = make_float4(fmaf(dec[k], run.x, off[k].x), fmaf(dec[k], run.y, off[k].y), fmaf(dec[k], run.z, off[k].z),
                                  fmaf(dec[k], run.w, off[k].w));
            }
        }
#pragma unroll
        for (int k = 0; k < SPB; ++k) {
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) dot[k] += __shfl_xor_sync(0xffffffffu, dot[k], o);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = dot[k];
        }
        __syncthreads();
        if (threadIdx.x < SPB) {
            const int c = c0 - (int)threadIdx.x;
            if (c >= 0 && c + 1 < d.nc) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < NTHR / 32; ++w) t += red[w][threadIdx.x];
                atomicAdd(dq + c, t);
            }
        }
        __syncthreads();
    }
    if (dinit && ok) reinterpret_cast<float4*>(dinit)[bh4] = run;
}
// element-wise fallback (P * N not a multiple of 4)
template <bool SEQ>
__global__ void __launch_bounds__(NTHR) state_pass_bwd_kernel_scalar(Dims d, Ws ws, float* dstates, float* dcsQ, const float* fin,
                                                                     const float* dfin, float* dinit) {
    __shared__ float red[NTHR / 32];
    const size_t PN = (size_t)d.P * d.N;
    const int nblk = (int)((PN + NTHR - 1) / NTHR);
    const int blk = blockIdx.x % nblk;
    const int h = (blockIdx.x / nblk) % d.H, b = blockIdx.x / (nblk * d.H);
    const size_t e = (size_t)blk * NTHR + threadIdx.x;
    const bool ok = e < PN;
    const size_t bh = ((size_t)b * d.H + h) * PN + e;   // this thread's element of a (batch, H, P, N) tensor
    float run = (dfin && ok) ? dfin[bh] : 0.f;
    for (int c = d.nc - 1; c >= 0; --c) {
        float* s = dstates + (((size_t)b * d.nc + c) * d.H + h) * PN + e;
        float off = 0.f;
        if (ok) {
            off = *s;
            *s = run;
        }
        float dot = 0.f;
        if (ok && c + 1 < d.nc) dot = run * ws.states[(((size_t)b * d.nc + c + 1) * d.H + h) * PN + e];
        else if (ok && dfin) dot = run * fin[bh];
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < NTHR / 32; ++w) t += red[w];
            if (c + 1 < d.nc || dfin) atomicAdd(dcsQ + ((size_t)b * d.H + h) * d.nc + c, t);
        }
        __syncthreads();
        const float csQ = ws.cs[(((size_t)b * d.H + h) * d.nc + c) * d.Q + d.Q - 1];
        const float dec = (SEQ && seq_end(d, b, c) != seq_prev(d, b, c)) ? 0.f : exp_acc(csQ);
        run = off + dec * run;
    }
    if (dinit && ok) dinit[bh] = run;
}

// ---- B3: Z = (CB o decay)^T dout + exp(cs_Q - cs) B G^T;  dx = dt' Z + D dout;
//          ddtp_exp[s] = sum_p x Z;  dcs_pos[l] = sum_p dout (out - D x);  dD += sum dout x --------
template <typename T, bool SEQ>
__global__ void __launch_bounds__(NTHR, 2) dx_kernel(View4<T> X, View4<T> Bv, View4<T> DO, View4<T> OUT, const float* D, Dims d, Ws ws,
                                                     const float* G, float* dx, OutS dxs, float* ddtp_exp, float* dcs_pos, float* dD, int x3,
                                                     int has_dfin) {
    Smem& sm = smem_ref();
    const int ntm = (d.Q + BM - 1) / BM, ntp = (d.P + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tp = bid % ntp; bid /= ntp;
    const int tm = bid % ntm; bid /= ntm;
    const int h = bid % d.H; bid /= d.H;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int g = h / d.hpg;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, p0 = tp * BN;
    if (m0 >= q) return;
    stage_cs(sm, 0, ws, d, b, h, c);
    if (SEQ) stage_sid(sm, d, b, c);
    __syncthreads();
    const float csQ = sm.cs[0][d.Q - 1];
    const int send_id = SEQ ? seq_end(d, b, c) : 0;
    const float* cb = ws.cb + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    const float* Gs = G + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N;
    const bool do_ifast = DO.s3 < DO.s1, b_ifast = Bv.s1 <= Bv.s3;
    Acc acc;
    acc.zero();
    int buf = 0;
    for (int k0 = (m0 / BK) * BK; k0 < q; k0 += BK, buf ^= 1) {  // l >= s
        fill_tile<BM, true>(sm.A[buf], true, [&](int i, int k) {
            const int s = m0 + i, l = k0 + k;
            if (SEQ && l < q && s <= l && sm.sid[l] != sm.sid[s]) return 0.f;
            return (l < q && s <= l) ? cb[(size_t)l * d.Q + s] * exp_acc(sm.cs[0][l] - sm.cs[0][s]) : 0.f;
        });
        fill_tile<BN, false>(sm.B[buf], do_ifast, [&](int i, int k) {
            const int p = p0 + i, l = k0 + k;
            return (p < d.P && l < q) ? DO.at(b, l0 + l, h, p) : 0.f;
        });
        __syncthreads();
        warp_mma<true, false>(acc, sm.A[buf], sm.B[buf], x3 != 0);
    }
    if (c + 1 < d.nc || has_dfin) {  // G of the last chunk is dfinal_states: zero unless given
        for (int k0 = 0; k0 < d.N; k0 += BK, buf ^= 1) {
            fill_tile<BM, true>(sm.A[buf], b_ifast, [&](int i, int k) {
                const int s = m0 + i, n = k0 + k;
                if (SEQ && s < q && sm.sid[s] != send_id) return 0.f;
                return (s < q && n < d.N) ? Bv.at(b, l0 + s, g, n) * exp_acc(csQ - sm.cs[0][s]) : 0.f;
            });
            fill_tile<BN, false>(sm.B[buf], false, [&](int i, int k) {
                const int p = p0 + i, n = k0 + k;
                return (p < d.P && n < d.N) ? Gs[(size_t)p * d.N + n] : 0.f;
            });
            __syncthreads();
            warp_mma<true, false>(acc, sm.A[buf], sm.B[buf], x3 != 0);
        }
    }
    const float Dh = D ? __ldg(D + h) : 0.f;
    // epilogue: each thread owns rows (g, g+8) of two m16 blocks; accumulate its row sums per row slot
    float r1[2][2] = {{0.f, 0.f}, {0.f, 0.f}}, r2[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    float dDl = 0.f;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int wm0 = (warp & 3) * 32, wn0 = (warp >> 2) * 32;
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int s = m0 + wm0 + mi * 16 + gq + ((r & 2) ? 8 : 0), p = p0 + wn0 + ni * 8 + 2 * tq + (r & 1);
                if (s < q && p < d.P) {
                    const float z = acc.v[mi][ni][r];
                    const float xv = X.at(b, l0 + s, h, p), dv = DO.at(b, l0 + s, h, p), ov = OUT.at(b, l0 + s, h, p);
                    dx[dxs.at(b, l0 + s, h, p)] = sm.dtp[0][s] * z + Dh * dv;
                    r1[mi][r >> 1] += xv * z;
                    r2[mi][r >> 1] += dv * (ov - Dh * xv);
                    dDl += dv * xv;
                }
            }
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            float a = r1[mi][hh], bb = r2[mi][hh];
            a += __shfl_xor_sync(0xffffffffu, a, 1); a += __shfl_xor_sync(0xffffffffu, a, 2);
            bb += __shfl_xor_sync(0xffffffffu, bb, 1); bb += __shfl_xor_sync(0xffffffffu, bb, 2);
            const int s = m0 + wm0 + mi * 16 + gq + hh * 8;
            if (tq == 0 && s < q) {
                const size_t off = (((size_t)b * d.H + h) * d.nc + c) * d.Q + s;
                atomicAdd(ddtp_exp + off, a);
                atomicAdd(dcs_pos + off, bb);
            }
        }
    if (dD) {
        const float tot = block_sum(sm, dDl);
        if (threadIdx.x == 0) atomicAdd(dD + h, tot);
    }
}

// B3 on the tcgen05 engine: same contractions, operands staged through registers (128-bit loads where the view
// allows) into UMMA tiles, accumulator row = one thread in the epilogue (row sums need no shuffles).
template <typename T, bool SEQ>
__global__ void __launch_bounds__(NTHR, TcEngine::MIN_CTAS) dx_kernel_tc(View4<T> X, View4<T> Bv, View4<T> DO, View4<T> OUT, const float* D, Dims d, Ws ws,
                                                        const float* G, float* dx, OutS dxs, float* ddtp_exp, float* dcs_pos, float* dD, int x3,
                                                        int has_dfin) {
    using E = TcEngine;
    E::Shared& sm = E::smem();
    const int ntm = (d.Q + BM - 1) / BM, ntp = (d.P + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tp = bid % ntp; bid /= ntp;
    const int tm = bid % ntm; bid /= ntm;
    const int h = bid % d.H; bid /= d.H;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int g = h / d.hpg;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, p0 = tp * BN;
    if (m0 >= q) return;
    stage_cs(sm, 0, ws, d, b, h, c);
    if (SEQ) stage_sid(sm, d, b, c);
    __syncthreads();
    const float csQ = sm.cs[0][d.Q - 1];
    const float* cb = ws.cb + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    const float* Gs = G + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N;
    E eng;
    eng.begin(sm);
    {   // Z += (CB o decay)^T dout : A(i = s, k = l) = CB[l][s] exp(cs_l - cs_s) for s <= l,  B(i = p, k = l) = dout[l][p]
        const int kb = (m0 / BK) * BK;
        const T* pdo = DO.p + b * DO.s0 + (int64_t)(l0 + kb) * DO.s1 + h * DO.s2 + (int64_t)p0 * DO.s3;
        const bool kib = DO.s3 == 1;
        eng.template pass<true, false>(
            sm, (q - kb + BK - 1) / BK, x3 != 0,
            [&](int kt, RegTile<BM>& r) { E::template load_any<BM>(r, cb + (size_t)(kb + kt * BK) * d.Q + m0, 1, d.Q, q - m0, q - kb - kt * BK, true); },
            [&](int kt, RegTile<BN>& r) { E::template load_any<BN>(r, pdo + (int64_t)kt * BK * DO.s1, DO.s3, DO.s1, d.P - p0, q - kb - kt * BK, kib); },
            [&](int kt, const RegTile<BM>& r, const tc::Dst& dst) {
                const int k0 = kb + kt * BK;
                E::template store_any<BM>(dst, r, true, [&](int i, int k, float v) {
                    const int sidx = m0 + i, l = k0 + k;
                    if (SEQ && l < q && sidx <= l && sm.sid[l] != sm.sid[sidx]) return 0.f;
                    return (l < q && sidx <= l) ? v * exp_acc(sm.cs[0][l] - sm.cs[0][sidx]) : 0.f;
                });
            },
            [&](int, const RegTile<BN>& r, const tc::Dst& dst) { E::template store_any<BN>(dst, r, kib, Identity()); });
    }
    if (c + 1 < d.nc || has_dfin) {   // Z += exp(cs_Q - cs_s) B G^T (G of the last chunk is dfinal_states: zero unless given)
        if (threadIdx.x < BM) {
            const int s = min(m0 + (int)threadIdx.x, d.Q - 1);
            sm.v1[0][threadIdx.x] = exp_acc(csQ - sm.cs[0][s]);
            if (SEQ && sm.sid[s] != seq_end(d, b, c)) sm.v1[0][threadIdx.x] = 0.f;
        }
        __syncthreads();
        const T* pbv = Bv.p + b * Bv.s0 + (int64_t)(l0 + m0) * Bv.s1 + g * Bv.s2;
        const bool kia = Bv.s1 == 1;
        eng.template pass<true, false>(
            sm, (d.N + BK - 1) / BK, x3 != 0,
            [&](int kt, RegTile<BM>& r) { E::template load_any<BM>(r, pbv + (int64_t)kt * BK * Bv.s3, Bv.s1, Bv.s3, q - m0, d.N - kt * BK, kia); },
            [&](int kt, RegTile<BN>& r) { E::template load_any<BN>(r, Gs + (size_t)p0 * d.N + kt * BK, d.N, 1, d.P - p0, d.N - kt * BK, false); },
            [&](int, const RegTile<BM>& r, const tc::Dst& dst) {
                E::template store_any<BM>(dst, r, kia, [&](int i, int, float v) { return v * sm.v1[0][i]; });
            },
            [&](int, const RegTile<BN>& r, const tc::Dst& dst) { E::template store_any<BN>(dst, r, false, Identity()); });
    }
    const float Dh = D ? __ldg(D + h) : 0.f;
    float r1 = 0.f, r2 = 0.f, dDl = 0.f;
    int srow = -1;
    eng.for_each(sm, [&](int m, int n, float& z) {
        const int sidx = m0 + m, pp = p0 + n;
        srow = sidx;
        if (sidx < q && pp < d.P) {
            const float xv = X.at(b, l0 + sidx, h, pp), dv = DO.at(b, l0 + sidx, h, pp), ov = OUT.at(b, l0 + sidx, h, pp);
            dx[dxs.at(b, l0 + sidx, h, pp)] = sm.dtp[0][sidx] * z + Dh * dv;
            r1 += xv * z;
            r2 += dv * (ov - Dh * xv);
            dDl += dv * xv;
        }
    });
    if (srow >= 0 && srow < q) {   // one thread = one row (its 32 columns)
        const size_t off = (((size_t)b * d.H + h) * d.nc + c) * d.Q + srow;
        atomicAdd(ddtp_exp + off, r1);
        atomicAdd(dcs_pos + off, r2);
    }
    if (dD) {
        const float tot = block_sum(sm, dDl);
        if (threadIdx.x == 0) atomicAdd(dD + h, tot);
    }
    eng.end(sm);
}

// ---- B4: dCB[l][s] = sum_{h in g} dt'_s exp(cs_l - cs_s) (dout_h x_h^T)[l, s],  s <= l ------------
template <typename T, bool SEQ>
__global__ void __launch_bounds__(NTHR, 2) dcb_kernel(View4<T> X, View4<T> DO, Dims d, Ws ws, float* dcb, int x3) {
    Smem& sm = smem_ref();
    const int ntm = (d.Q + BM - 1) / BM, ntn = (d.Q + BN - 1) / BN;
    int bid = blockIdx.x;
    const int tn = bid % ntn; bid /= ntn;
    const int tm = bid % ntm; bid /= ntm;
    const int g = bid % d.G; bid /= d.G;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, s0 = tn * BN;
    if (m0 >= q || s0 >= q || s0 > m0 + BM - 1) return;
    const bool do_ifast = DO.s1 <= DO.s3, x_ifast = X.s1 <= X.s3;
    if (SEQ) stage_sid(sm, d, b, c);   // read after the barrier of the first head's staging
    Acc tot;
    tot.zero();
    int buf = 0;
    for (int hh = 0; hh < d.hpg; ++hh) {
        const int h = g * d.hpg + hh, hb = hh & 1;
        stage_cs(sm, hb, ws, d, b, h, c);
        __syncthreads();
        Acc acc;
        acc.zero();
        for (int k0 = 0; k0 < d.P; k0 += BK, buf ^= 1) {
            fill_tile<BM, true>(sm.A[buf], do_ifast, [&](int i, int k) {
                const int l = m0 + i, p = k0 + k;
                return (l < q && p < d.P) ? DO.at(b, l0 + l, h, p) : 0.f;
            });
            fill_tile<BN, true>(sm.B[buf], x_ifast, [&](int i, int k) {
                const int s = s0 + i, p = k0 + k;
                return (s < q && p < d.P) ? X.at(b, l0 + s, h, p) : 0.f;
            });
            __syncthreads();
            warp_mma<true, true>(acc, sm.A[buf], sm.B[buf], x3 != 0);
        }
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int gq = lane >> 2, tq = lane & 3;
        const int wm0 = (warp & 3) * 32, wn0 = (warp >> 2) * 32;
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int l = m0 + wm0 + mi * 16 + gq + ((r & 2) ? 8 : 0), s = s0 + wn0 + ni * 8 + 2 * tq + (r & 1);
                    if (l < q && s <= l && (!SEQ || sm.sid[l] == sm.sid[s])) tot.v[mi][ni][r] += sm.dtp[hb][s] * exp_acc(sm.cs[hb][l] - sm.cs[hb][s]) * acc.v[mi][ni][r];
                }
    }
    float* o = dcb + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    for_each_acc(tot, [&](int m, int n, float& v) {
        const int l = m0 + m, s = s0 + n;
        if (l < q && s < q) o[(size_t)l * d.Q + s] = v;
    });
}

// ---- B5: dC = dCB B + sum_h exp(cs_h) dout_h Sin_h ;  dB = dCB^T C + sum_h exp(cs_Q - cs) dt' x_h G_h ----
template <typename T, bool SEQ>
__global__ void __launch_bounds__(NTHR, 2) dbc_kernel(View4<T> X, View4<T> Bv, View4<T> Cv, View4<T> DO, Dims d, Ws ws,
                                                      const float* dcb_all, const float* G, float* dB, float* dC, OutS dbs, OutS dcs, int x3,
                                                      int has_dfin) {
    Smem& sm = smem_ref();
    const int ntm = (d.Q + BM - 1) / BM, ntn = (d.N + BN - 1) / BN;
    int bid = blockIdx.x;
    const int which = bid & 1; bid >>= 1;  // 0: dC, 1: dB
    const int tn = bid % ntn; bid /= ntn;
    const int tm = bid % ntm; bid /= ntm;
    const int g = bid % d.G; bid /= d.G;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, n0 = tn * BN;
    if (m0 >= q) return;
    const float* dcb = dcb_all + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    Acc acc;
    acc.zero();
    int buf = 0;
    if (which == 0) {
        const bool b_ifast = Bv.s3 < Bv.s1;
        const int send = min(q, m0 + BM);
        for (int k0 = 0; k0 < send; k0 += BK, buf ^= 1) {
            fill_tile<BM, false>(sm.A[buf], false, [&](int i, int k) {
                const int l = m0 + i, s = k0 + k;
                return (l < q && s <= l) ? dcb[(size_t)l * d.Q + s] : 0.f;
            });
            fill_tile<BN, false>(sm.B[buf], b_ifast, [&](int i, int k) {
                const int n = n0 + i, s = k0 + k;
                return (n < d.N && s < q) ? Bv.at(b, l0 + s, g, n) : 0.f;
            });
            __syncthreads();
            warp_mma<false, false>(acc, sm.A[buf], sm.B[buf], x3 != 0);
        }
    } else {
        const bool c_ifast = Cv.s3 < Cv.s1;
        for (int k0 = (m0 / BK) * BK; k0 < q; k0 += BK, buf ^= 1) {
            fill_tile<BM, true>(sm.A[buf], true, [&](int i, int k) {
                const int s = m0 + i, l = k0 + k;
                return (l < q && s <= l) ? dcb[(size_t)l * d.Q + s] : 0.f;
            });
            fill_tile<BN, false>(sm.B[buf], c_ifast, [&](int i, int k) {
                const int n = n0 + i, l = k0 + k;
                return (n < d.N && l < q) ? Cv.at(b, l0 + l, g, n) : 0.f;
            });
            __syncthreads();
            warp_mma<true, false>(acc, sm.A[buf], sm.B[buf], x3 != 0);
        }
    }
    // state terms, head by head (K = p)
    const View4<T>& Asrc = which == 0 ? DO : X;
    const bool a_ifast = Asrc.s1 <= Asrc.s3;
    const float* Sbase = which == 0 ? ws.states : G;
    if (which == 0 || c + 1 < d.nc || has_dfin) {   // dB: G of the last chunk is dfinal_states, zero unless given
        // dC: only positions of the sequence entering the chunk see Sin; dB: only those of the sequence open at its end feed G
        const int ref = SEQ ? (which == 0 ? seq_prev(d, b, c) : seq_end(d, b, c)) : 0;
        if (SEQ) stage_sid(sm, d, b, c);
        for (int hh = 0; hh < d.hpg; ++hh) {
            const int h = g * d.hpg + hh, hb = hh & 1;
            stage_cs(sm, hb, ws, d, b, h, c);
            __syncthreads();
            const float csQ = sm.cs[hb][d.Q - 1];
            const float* S = Sbase + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N;
            for (int k0 = 0; k0 < d.P; k0 += BK, buf ^= 1) {
                fill_tile<BM, true>(sm.A[buf], a_ifast, [&](int i, int k) {
                    const int l = m0 + i, p = k0 + k;
                    if (l >= q || p >= d.P) return 0.f;
                    if (SEQ && sm.sid[l] != ref) return 0.f;
                    const float w = which == 0 ? exp_acc(sm.cs[hb][l]) : exp_acc(csQ - sm.cs[hb][l]) * sm.dtp[hb][l];
                    return Asrc.at(b, l0 + l, h, p) * w;
                });
                fill_tile<BN, true>(sm.B[buf], true, [&](int i, int k) {
                    const int n = n0 + i, p = k0 + k;
                    return (n < d.N && p < d.P) ? S[(size_t)p * d.N + n] : 0.f;
                });
                __syncthreads();
                warp_mma<true, true>(acc, sm.A[buf], sm.B[buf], x3 != 0);
            }
        }
    }
    float* o = which == 0 ? dC : dB;
    const OutS os = which == 0 ? dcs : dbs;
    for_each_acc(acc, [&](int m, int n, float& v) {
        const int l = m0 + m, nn = n0 + n;
        if (l < q && nn < d.N) o[os.at(b, l0 + l, g, nn)] = v;
    });
}

// B5 on the tcgen05 engine.
template <typename T>
__global__ void __launch_bounds__(NTHR, TcEngine::MIN_CTAS) dbc_kernel_tc(View4<T> X, View4<T> Bv, View4<T> Cv, View4<T> DO, Dims d, Ws ws,
                                                         const float* dcb_all, const float* G, float* dB, float* dC, OutS dbs, OutS dcs, int x3,
                                                         int has_dfin) {
    using E = TcEngine;
    E::Shared& sm = E::smem();
    const int ntm = (d.Q + BM - 1) / BM, ntn = (d.N + BN - 1) / BN;
    int bid = blockIdx.x;
    const int which = bid & 1; bid >>= 1;  // 0: dC, 1: dB
    const int tn = bid % ntn; bid /= ntn;
    const int tm = bid % ntm; bid /= ntm;
    const int g = bid % d.G; bid /= d.G;
    const int c = bid % d.nc;
    const int b = bid / d.nc;
    const int q = min(d.Q, d.L - c * d.Q), l0 = c * d.Q;
    const int m0 = tm * BM, n0 = tn * BN;
    if (m0 >= q) return;
    const float* dcb = dcb_all + (((size_t)b * d.nc + c) * d.G + g) * (size_t)d.Q * d.Q;
    E eng;
    eng.begin(sm);
    if (which == 0) {   // dC[l][n] += sum_{s <= l} dCB[l][s] B[s][n]:  A(i = l, k = s),  B(i = n, k = s)
        const int send = min(q, m0 + BM);
        const T* pb = Bv.p + b * Bv.s0 + (int64_t)l0 * Bv.s1 + g * Bv.s2 + (int64_t)n0 * Bv.s3;
        const bool kib = Bv.s3 == 1;
        eng.template pass<false, false>(
            sm, (send + BK - 1) / BK, x3 != 0,
            [&](int kt, RegTile<BM>& r) { E::template load_any<BM>(r, dcb + (size_t)m0 * d.Q + kt * BK, d.Q, 1, q - m0, send - kt * BK, false); },
            [&](int kt, RegTile<BN>& r) { E::template load_any<BN>(r, pb + (int64_t)kt * BK * Bv.s1, Bv.s3, Bv.s1, d.N - n0, q - kt * BK, kib); },
            [&](int kt, const RegTile<BM>& r, const tc::Dst& dst) {
                const int k0 = kt * BK;
                E::template store_any<BM>(dst, r, false, [&](int i, int k, float v) { return (k0 + k <= m0 + i) ? v : 0.f; });
            },
            [&](int, const RegTile<BN>& r, const tc::Dst& dst) { E::template store_any<BN>(dst, r, kib, Identity()); });
    } else {            // dB[s][n] += sum_{l >= s} dCB[l][s] C[l][n]:  A(i = s, k = l),  B(i = n, k = l)
        const int kb = (m0 / BK) * BK;
        const T* pc = Cv.p + b * Cv.s0 + (int64_t)(l0 + kb) * Cv.s1 + g * Cv.s2 + (int64_t)n0 * Cv.s3;
        const bool kib = Cv.s3 == 1;
        eng.template pass<true, false>(
            sm, (q - kb + BK - 1) / BK, x3 != 0,
            [&](int kt, RegTile<BM>& r) { E::template load_any<BM>(r, dcb + (size_t)(kb + kt * BK) * d.Q + m0, 1, d.Q, q - m0, q - kb - kt * BK, true); },
            [&](int kt, RegTile<BN>& r) { E::template load_any<BN>(r, pc + (int64_t)kt * BK * Cv.s1, Cv.s3, Cv.s1, d.N - n0, q - kb - kt * BK, kib); },
            [&](int kt, const RegTile<BM>& r, const tc::Dst& dst) {
                const int k0 = kb + kt * BK;
                E::template store_any<BM>(dst, r, true, [&](int i, int k, float v) { return (m0 + i <= k0 + k) ? v : 0.f; });
            },
            [&](int, const RegTile<BN>& r, const tc::Dst& dst) { E::template store_any<BN>(dst, r, kib, Identity()); });
    }
    // state terms, head by head (K = p):  A(i = l, k = p) = src[l][p] w_l,  B(i = n, k = p) = S[p][n]
    const View4<T>& Asrc = which == 0 ? DO : X;
    const float* Sbase = which == 0 ? ws.states : G;
    if (which == 0 || c + 1 < d.nc || has_dfin) {   // dB: G of the last chunk is dfinal_states, zero unless given
        const bool kia = Asrc.s1 == 1;
        for (int hh = 0; hh < d.hpg; ++hh) {
            const int h = g * d.hpg + hh, hb = hh & 1;
            stage_cs(sm, hb, ws, d, b, h, c);
            __syncthreads();
            const float csQ = sm.cs[hb][d.Q - 1];
            if (threadIdx.x < BM) {   // the row factor, once per (head, row) instead of once per element
                const int l = min(m0 + (int)threadIdx.x, d.Q - 1);
                sm.v1[hb][threadIdx.x] = which == 0 ? exp_acc(sm.cs[hb][l]) : exp_acc(csQ - sm.cs[hb][l]) * sm.dtp[hb][l];
                // dC: only positions of the sequence entering the chunk see Sin; dB: only those of the sequence open at its end feed G
                if (d.seq.p && seq_at(d, b, c, l) != (which == 0 ? seq_prev(d, b, c) : seq_end(d, b, c))) sm.v1[hb][threadIdx.x] = 0.f;
            }
            __syncthreads();
            const float* S = Sbase + (((size_t)b * d.nc + c) * d.H + h) * (size_t)d.P * d.N;
            const T* pa = Asrc.p + b * Asrc.s0 + (int64_t)(l0 + m0) * Asrc.s1 + h * Asrc.s2;
            eng.template pass<true, true>(
                sm, (d.P + BK - 1) / BK, x3 != 0,
                [&](int kt, RegTile<BM>& r) { E::template load_any<BM>(r, pa + (int64_t)kt * BK * Asrc.s3, Asrc.s1, Asrc.s3, q - m0, d.P - kt * BK, kia); },
                [&](int kt, RegTile<BN>& r) { E::template load_any<BN>(r, S + (size_t)kt * BK * d.N + n0, 1, d.N, d.N - n0, d.P - kt * BK, true); },
                [&](int, const RegTile<BM>& r, const tc::Dst& dst) {
                    E::template store_any<BM>(dst, r, kia, [&](int i, int, float v) { return v * sm.v1[hb][i]; });
                },
                [&](int, const RegTile<BN>& r, const tc::Dst& dst) { E::template store_any<BN>(dst, r, true, Identity()); });
        }
    }
    float* o = which == 0 ? dC : dB;
    const OutS os = which == 0 ? dcs : dbs;
    eng.for_each(sm, [&](int m, int n, float& v) {
        const int l = m0 + m, nn = n0 + n;
        if (l < q && nn < d.N) o[os.at(b, l0 + l, g, nn)] = v;
    });
    eng.end(sm);
}

// ---- B6: d cs -> d(dt' A) (reverse cumsum) -> ddt', dA, ddt, ddt_bias ----------------------------
template <typename T>
__global__ void __launch_bounds__(MAXQ) dt_bwd_kernel(const T* dt, int64_t s0, int64_t s1, int64_t s2, const float* A,
                                                      const float* dt_bias, int softplus, float dt_min, float dt_max, Dims d, Ws ws,
                                                      const float* ddtp_exp, const float* dcs_pos, const float* dcsQ, float* ddt, OutS dts,
                                                      float* dA, float* ddt_bias) {
    __shared__ float wsum[MAXQ / 32];
    __shared__ float red[2][MAXQ / 32];
    const int c = blockIdx.x % d.nc, h = (blockIdx.x / d.nc) % d.H, b = blockIdx.x / (d.nc * d.H);
    const int i = threadIdx.x, l = c * d.Q + i;
    const size_t off = (((size_t)b * d.H + h) * d.nc + c) * d.Q + i;
    const bool in = i < d.Q;
    const float dtp = in ? ws.dtp[off] : 0.f;
    const float de = in ? ddtp_exp[off] : 0.f;
    float x = in ? dcs_pos[off] - dtp * de : 0.f;
    if (i == d.Q - 1) x += dcsQ[((size_t)b * d.H + h) * d.nc + c];
    // inclusive suffix sum over the chunk
    const int lane = i & 31, w = i >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_down_sync(0xffffffffu, x, o);
        if (lane + o < 32) x += y;
    }
    if (lane == 0) wsum[w] = x;
    __syncthreads();
    float post = 0.f;
    for (int j = w + 1; j < MAXQ / 32; ++j) post += (j * 32 < blockDim.x) ? wsum[j] : 0.f;
    const float ddA = x + post;
    const float Ah = __ldg(A + h);
    const float ddtp = de + ddA * Ah;
    float dAl = ddA * dtp, g = 0.f;
    if (in && l < d.L) {
        const float raw = to_f32<T>(__ldg(dt + b * s0 + l * s1 + h * s2)) + (dt_bias ? __ldg(dt_bias + h) : 0.f);
        float v = raw, dv = 1.f;
        if (softplus) {
            v = softplus20(raw);
            dv = raw > 20.f ? 1.f : 1.f / (1.f + expf(-raw));
        }
        if (v < dt_min || v > dt_max) dv = 0.f;
        g = ddtp * dv;
        ddt[dts.at(b, l, h, 0)] = g;
    } else {
        dAl = 0.f;
    }
    float r0 = dAl, r1 = g;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        r0 += __shfl_xor_sync(0xffffffffu, r0, o);
        r1 += __shfl_xor_sync(0xffffffffu, r1, o);
    }
    if (lane == 0) { red[0][w] = r0; red[1][w] = r1; }
    __syncthreads();
    if (i == 0) {
        float t0 = 0.f, t1 = 0.f;
        for (int j = 0; j < (int)blockDim.x / 32; ++j) { t0 += red[0][j]; t1 += red[1][j]; }
        atomicAdd(dA + h, t0);
        if (ddt_bias) atomicAdd(ddt_bias + h, t1);
    }
}

// ---- V1: state after the last token of each packed sequence (batch 1), after the forward -----------------------------
// e = the sequence's last position, c its chunk:  S = sum_{s in [max(start, c Q), e]} exp(cs_e - cs_s) dt'_s x_s B_s^T
//                                                   + exp(cs_e) Sin[c]   when the sequence began before chunk c (or at 0)
// (mamba_ssm's chunk_state_varlen adds Sin[c] only when it began before chunk c, so it leaves initial_states out of a first
// sequence that ends inside chunk 0; here that sequence includes them, as out and final_states do)
// Grid (nseq, H, P N / 256); one thread per (p, n), SIMT over the at most Q tail positions.
template <typename T>
__global__ void __launch_bounds__(NTHR) varlen_states_kernel(View4<T> X, View4<T> Bv, Dims d, Ws ws, const int32_t* cu_seqlens, float* states) {
    __shared__ float w[MAXQ];
    const int k = blockIdx.x, h = blockIdx.y, g = h / d.hpg;
    const int start = min(max(__ldg(cu_seqlens + k), 0), d.L), end = min(max(__ldg(cu_seqlens + k + 1), 0), d.L);
    const int e = end - 1, c = max(e, 0) / d.Q, l0 = c * d.Q, s0 = max(start, l0);
    const size_t csoff = ((size_t)h * d.nc + c) * d.Q;
    const float cse = end > start ? ws.cs[csoff + e - l0] : 0.f;
    for (int i = threadIdx.x; i < d.Q; i += NTHR) {
        const int s = l0 + i;
        w[i] = (s >= s0 && s <= e) ? exp_acc(cse - ws.cs[csoff + i]) * ws.dtp[csoff + i] : 0.f;
    }
    __syncthreads();
    const int PN = d.P * d.N, idx = blockIdx.z * NTHR + threadIdx.x;
    if (idx >= PN) return;
    const int p = idx / d.N, n = idx % d.N;
    float acc = 0.f;
    if (end > start) {
        // the chunk-entry state belongs to this sequence when it began before the chunk (or is the row's first); with seq_idx
        // the forward's own mask decides, so out, final_states and these states agree
        const bool entry = (start < l0 || start == 0) && (!d.seq.p || d.seq.at(0, e) == seq_prev(d, 0, c));
        if (entry) acc = exp_acc(cse) * ws.states[((size_t)c * d.H + h) * PN + idx];
        for (int s = s0; s <= e; ++s) acc = fmaf(w[s - l0] * X.at(0, s, h, p), Bv.at(0, s, g, n), acc);
    }
    states[((size_t)k * d.H + h) * PN + idx] = acc;
}

// ---- gated RMSNorm (SSD/MedSSD.py:393-394): y = rmsnorm(x silu(z)) w ------------------------------
__device__ __forceinline__ float silu_f(float z) { return z / (1.f + expf(-z)); }

__global__ void __launch_bounds__(256) rmsnorm_gated_fwd_kernel(const float* x, const float* z, const float* w, float* y, float* rstd,
                                                                int64_t rows, int dim, float eps) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const float* xr = x + row * dim;
    const float* zr = z + row * dim;
    float ss = 0.f;
    for (int i = lane; i < dim; i += 32) {
        const float v = xr[i] * silu_f(zr[i]);
        ss += v * v;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float r = rsqrtf(ss / dim + eps);
    if (lane == 0) rstd[row] = r;
    float* yr = y + row * dim;
    for (int i = lane; i < dim; i += 32) yr[i] = xr[i] * silu_f(zr[i]) * r * __ldg(w + i);
}

// dw_partial is (gridDim.x, dim): block-local sums over the block's rows (the host adds the rows up)
__global__ void __launch_bounds__(256) rmsnorm_gated_bwd_kernel(const float* x, const float* z, const float* w, const float* rstd,
                                                                const float* dy, float* dx, float* dz, float* dw_partial,
                                                                int64_t rows, int dim, int rows_per_block) {
    extern __shared__ float dw_s[];  // dim floats
    for (int i = threadIdx.x; i < dim; i += 256) dw_s[i] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r_end = r_begin + rows_per_block < rows ? r_begin + rows_per_block : rows;
    for (int64_t row = r_begin + warp; row < r_end; row += 8) {
        const float* xr = x + row * dim;
        const float* zr = z + row * dim;
        const float* gr = dy + row * dim;
        const float r = rstd[row];
        float dot = 0.f;
        for (int i = lane; i < dim; i += 32) {
            const float vh = xr[i] * silu_f(zr[i]) * r;
            dot += gr[i] * __ldg(w + i) * vh;
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        const float mean = dot / dim;
        for (int i = lane; i < dim; i += 32) {
            const float zz = zr[i], xx = xr[i];
            const float sg = 1.f / (1.f + expf(-zz));
            const float sl = zz * sg;
            const float vh = xx * sl * r;
            const float gy = gr[i];
            const float dv = r * (gy * __ldg(w + i) - vh * mean);
            dx[row * dim + i] = dv * sl;
            dz[row * dim + i] = dv * xx * sg * (1.f + zz * (1.f - sg));
            atomicAdd(&dw_s[i], gy * vh);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < dim; i += 256) dw_partial[(size_t)blockIdx.x * dim + i] = dw_s[i];
}

// ---- host side ----------------------------------------------------------------------------------
static int validate(const b200_ssd_fwd_params* p) {
    B200_REQUIRE(p != nullptr, "b200_ssd: params is NULL");
    B200_REQUIRE(p->batch > 0 && p->seqlen > 0 && p->nheads > 0 && p->headdim > 0 && p->dstate > 0,
                 "b200_ssd: batch/seqlen/nheads/headdim/dstate must be positive (got %d/%d/%d/%d/%d)", p->batch, p->seqlen,
                 p->nheads, p->headdim, p->dstate);
    B200_REQUIRE(p->n_groups >= 1 && p->nheads % p->n_groups == 0, "b200_ssd: nheads %d is not divisible by n_groups %d", p->nheads,
                 p->n_groups);
    B200_REQUIRE(p->chunk_size >= 32 && p->chunk_size <= MAXQ && p->chunk_size % 32 == 0,
                 "b200_ssd: chunk_size %d must be a multiple of 32 in [32, %d]", p->chunk_size, MAXQ);
    B200_REQUIRE(p->io_dtype >= B200_F32 && p->io_dtype <= B200_F16, "b200_ssd: bad io_dtype %d", p->io_dtype);
    B200_REQUIRE(p->x && p->dt && p->A && p->B && p->C, "b200_ssd: x/dt/A/B/C must be non-NULL");
    B200_REQUIRE(p->workspace != nullptr, "b200_ssd: workspace is NULL");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(p->workspace) & 15) == 0, "b200_ssd: workspace must be 16-byte aligned");
    B200_REQUIRE(p->seq_idx == nullptr || (p->seq_idx_stride[0] >= 0 && p->seq_idx_stride[1] >= 0),
                 "b200_ssd: seq_idx strides must be non-negative (got %lld, %lld)", (long long)p->seq_idx_stride[0],
                 (long long)p->seq_idx_stride[1]);
    return 0;
}

template <class K>
static int set_smem(K kernel, size_t bytes = sizeof(Smem)) {
    bytes = sizeof(tc::Shared) > sizeof(Smem) ? sizeof(tc::Shared) : sizeof(Smem);   // upper bound only; occupancy follows the launch's size
    const cudaError_t e = func_attr_per_device((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);   // per (kernel, device)
    if (e != cudaSuccess) {
        set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}

#define LAUNCH(kernel, grid, block, smem, st, ...)                  \
    do {                                                            \
        if ((smem) > 0)                                             \
            if (int rc_ = set_smem(kernel, (smem))) return rc_;     \
        kernel<<<(unsigned)(grid), (block), (smem), (st)>>>(__VA_ARGS__); \
        if (int rc_ = check_launch(#kernel)) return rc_;            \
    } while (0)

// tcgen05 / TMEM engine for the forward contractions (B200_SSD_TC=0 selects the mma.sync tiles)
static bool use_tcgen05() {
    static const bool on = [] {
        const char* e = getenv("B200_SSD_TC");
        return !(e && e[0] == '0');
    }();
    return on;
}

// K2 + K3: chunk states, then state passing (chunk-entry states and final_states)
template <typename T, bool SEQ>
static int states_fwd(const b200_ssd_fwd_params* p, const Dims& d, const Ws& ws, const View4<T>& X, const View4<T>& Bv, size_t smem, bool tcg,
                      cudaStream_t st) {
    const int x3 = p->precision == 0;
    const size_t grid = (size_t)d.batch * d.nc * d.H * ((d.P + BN - 1) / BN) * ((d.N + BM - 1) / BM);
    if (tcg) LAUNCH((chunk_state_kernel<T, 0, TcEngine, SEQ>), grid, NTHR, smem, st, X, Bv, d, ws, ws.states, x3);
    else LAUNCH((chunk_state_kernel<T, 0, MmaEngine, SEQ>), grid, NTHR, smem, st, X, Bv, d, ws, ws.states, x3);
    const size_t PN = (size_t)d.P * d.N;
    const bool vec = PN % 4 == 0 && ((uintptr_t)ws.states & 15) == 0 && ((uintptr_t)p->initial_states & 15) == 0 &&
                     ((uintptr_t)p->final_states & 15) == 0 && (size_t)d.batch * d.H <= 65535;
    if (vec) {
        state_pass_kernel<SEQ><<<dim3((unsigned)((PN / 4 + 255) / 256), (unsigned)(d.batch * d.H)), 256, 0, st>>>(d, ws, p->initial_states,
                                                                                                         p->final_states);
        if (int rc_ = check_launch("state_pass_kernel")) return rc_;
    } else {
        const size_t n = (size_t)d.batch * d.H * PN;
        LAUNCH(state_pass_kernel_scalar<SEQ>, (n + 255) / 256, 256, 0, st, d, ws, p->initial_states, p->final_states);
    }
    return 0;
}

template <typename T, class E>
static int chunk_scan(const b200_ssd_fwd_params* p, const Dims& d, const Ws& ws, const View4<T>& X, const View4<T>& Cv, size_t smem,
                      cudaStream_t st) {
    const size_t grid = (size_t)d.batch * d.nc * d.H * ((d.Q + BM - 1) / BM) * ((d.P + BN - 1) / BN);
    const int x3 = p->precision == 0, has_init = p->initial_states != nullptr;
    if (d.seq.p)
        LAUNCH((chunk_scan_kernel<T, E, true>), grid, NTHR, smem, st, X, Cv, p->D, d, ws, (T*)p->out, p->out_stride[0], p->out_stride[1],
               p->out_stride[2], p->out_stride[3], has_init, x3);
    else
        LAUNCH((chunk_scan_kernel<T, E, false>), grid, NTHR, smem, st, X, Cv, p->D, d, ws, (T*)p->out, p->out_stride[0], p->out_stride[1],
               p->out_stride[2], p->out_stride[3], has_init, x3);
    return 0;
}

template <typename T>
static int fwd_impl(const b200_ssd_fwd_params* p, cudaStream_t st) {
    const Dims d = make_dims(*p);
    const Ws ws = make_ws(p->workspace, d);
    const View4<T> X = view4<T>(p->x, p->x_stride), Bv = view4<T>(p->B, p->B_stride), Cv = view4<T>(p->C, p->C_stride);
    const int x3 = p->precision == 0;
    const size_t SM = sizeof(Smem);
    const int ntq128 = (d.Q + BM - 1) / BM, ntq64 = (d.Q + BN - 1) / BN;
    LAUNCH((dt_cumsum_kernel<T>), (size_t)d.batch * d.H * d.nc, d.Q, 0, st, (const T*)p->dt, p->dt_stride[0], p->dt_stride[1],
           p->dt_stride[2], p->A, p->dt_bias, p->dt_softplus, p->dt_min, p->dt_max, d, ws);
    const bool tcg = use_tcgen05();
    const size_t SMT = x3 ? tc::SMEM_X3 : tc::SMEM_TF32;
    if (d.seq.p) {
        if (int rc = states_fwd<T, true>(p, d, ws, X, Bv, tcg ? SMT : SM, tcg, st)) return rc;
    } else {
        if (int rc = states_fwd<T, false>(p, d, ws, X, Bv, tcg ? SMT : SM, tcg, st)) return rc;
    }
    if (tcg) {
        LAUNCH((cb_kernel<T, TcEngine>), (size_t)d.batch * d.nc * d.G * ntq128 * ntq64, NTHR, SMT, st, Cv, Bv, d, ws, x3);
        return chunk_scan<T, TcEngine>(p, d, ws, X, Cv, SMT, st);
    }
    LAUNCH((cb_kernel<T, MmaEngine>), (size_t)d.batch * d.nc * d.G * ntq128 * ntq64, NTHR, SM, st, Cv, Bv, d, ws, x3);
    return chunk_scan<T, MmaEngine>(p, d, ws, X, Cv, SM, st);
}

struct Scratch {
    float* dstates;   // [b][nc][h][P][N]
    float* dcb;       // [b][nc][g][Q][Q]
    float* ddtp_exp;  // [b][h][nc][Q]
    float* dcs_pos;   // [b][h][nc][Q]
    float* dcsQ;      // [b][h][nc]
};
static size_t scratch_zero_floats(const Dims& d) { return 2 * ws_dt_floats(d) + (size_t)d.batch * d.H * d.nc; }
static Scratch make_scratch(float* base, const Dims& d) {
    Scratch s;
    s.ddtp_exp = base;  // the three atomically-accumulated arrays first: one memset covers them
    s.dcs_pos = s.ddtp_exp + ws_dt_floats(d);
    s.dcsQ = s.dcs_pos + ws_dt_floats(d);
    size_t off = scratch_zero_floats(d);
    off = (off + 3) & ~(size_t)3;
    s.dstates = base + off;
    s.dcb = s.dstates + ws_state_floats(d);
    return s;
}

// B1 - B5 (B6, dt_bwd_kernel, needs no mask: the masked terms are already absent from its inputs)
template <typename T, bool SEQ>
static int bwd_masked(const b200_ssd_bwd_params* q, const Dims& d, const Ws& ws, const Scratch& sc, const View4<T>& X, const View4<T>& Bv,
                      const View4<T>& Cv, const View4<T>& DO, const View4<T>& OUT, const OutS& dxs, const OutS& dbs, const OutS& dcs,
                      cudaStream_t st) {
    const b200_ssd_fwd_params* p = &q->f;
    const int x3 = p->precision == 0;
    const size_t SM = sizeof(Smem);
    const int ntq128 = (d.Q + BM - 1) / BM, ntq64 = (d.Q + BN - 1) / BN;
    const int ntn128 = (d.N + BM - 1) / BM, ntn64 = (d.N + BN - 1) / BN, ntp64 = (d.P + BN - 1) / BN;
    if (use_tcgen05())
        LAUNCH((chunk_state_kernel<T, 1, TcEngine, SEQ>), (size_t)d.batch * d.nc * d.H * ntp64 * ntn128, NTHR, (x3 ? tc::SMEM_X3 : tc::SMEM_TF32),
               st, DO, Cv, d, ws, sc.dstates, x3);
    else
        LAUNCH((chunk_state_kernel<T, 1, MmaEngine, SEQ>), (size_t)d.batch * d.nc * d.H * ntp64 * ntn128, NTHR, SM, st, DO, Cv, d, ws, sc.dstates,
               x3);
    const int has_dfin = q->dfinal_states != nullptr;
    {
        const size_t PN = (size_t)d.P * d.N;
        const bool vec = PN % 4 == 0 && ((uintptr_t)ws.states & 15) == 0 && ((uintptr_t)sc.dstates & 15) == 0 &&
                         ((uintptr_t)q->final_states & 15) == 0 && ((uintptr_t)q->dfinal_states & 15) == 0 &&
                         ((uintptr_t)q->dinitial_states & 15) == 0 && (size_t)d.batch * d.H <= 65535;
        if (vec) {
            state_pass_bwd_kernel<SEQ><<<dim3((unsigned)((PN / 4 + NTHR - 1) / NTHR), (unsigned)(d.batch * d.H)), NTHR, 0, st>>>(
                d, ws, sc.dstates, sc.dcsQ, q->final_states, q->dfinal_states, q->dinitial_states);
            if (int rc_ = check_launch("state_pass_bwd_kernel")) return rc_;
        } else {
            const int nblk = (int)((PN + NTHR - 1) / NTHR);
            LAUNCH(state_pass_bwd_kernel_scalar<SEQ>, (size_t)d.batch * d.H * nblk, NTHR, 0, st, d, ws, sc.dstates, sc.dcsQ, q->final_states,
                   q->dfinal_states, q->dinitial_states);
        }
    }
    if (use_tcgen05())
        LAUNCH((dx_kernel_tc<T, SEQ>), (size_t)d.batch * d.nc * d.H * ntq128 * ntp64, NTHR, (x3 ? tc::SMEM_X3 : tc::SMEM_TF32), st, X, Bv, DO, OUT,
               p->D, d, ws, sc.dstates, q->dx, dxs, sc.ddtp_exp, sc.dcs_pos, q->dD, x3, has_dfin);
    else
        LAUNCH((dx_kernel<T, SEQ>), (size_t)d.batch * d.nc * d.H * ntq128 * ntp64, NTHR, SM, st, X, Bv, DO, OUT, p->D, d, ws, sc.dstates, q->dx,
               dxs, sc.ddtp_exp, sc.dcs_pos, q->dD, x3, has_dfin);
    LAUNCH((dcb_kernel<T, SEQ>), (size_t)d.batch * d.nc * d.G * ntq128 * ntq64, NTHR, SM, st, X, DO, d, ws, sc.dcb, x3);
    if (use_tcgen05())
        LAUNCH((dbc_kernel_tc<T>), (size_t)d.batch * d.nc * d.G * ntq128 * ntn64 * 2, NTHR, (x3 ? tc::SMEM_X3 : tc::SMEM_TF32), st, X, Bv, Cv, DO, d,
               ws, sc.dcb, sc.dstates, q->dB, q->dC, dbs, dcs, x3, has_dfin);
    else
        LAUNCH((dbc_kernel<T, SEQ>), (size_t)d.batch * d.nc * d.G * ntq128 * ntn64 * 2, NTHR, SM, st, X, Bv, Cv, DO, d, ws, sc.dcb, sc.dstates,
               q->dB, q->dC, dbs, dcs, x3, has_dfin);
    return 0;
}

template <typename T>
static int bwd_impl(const b200_ssd_bwd_params* q, cudaStream_t st) {
    const b200_ssd_fwd_params* p = &q->f;
    const Dims d = make_dims(*p);
    const Ws ws = make_ws(p->workspace, d);
    const Scratch sc = make_scratch(q->scratch, d);
    const View4<T> X = view4<T>(p->x, p->x_stride), Bv = view4<T>(p->B, p->B_stride), Cv = view4<T>(p->C, p->C_stride);
    const View4<T> DO = view4<T>(q->dout, q->dout_stride), OUT = view4<T>(p->out, p->out_stride);
    const OutS dxs = outs_of(q->dx_stride, d.L, d.H, d.P), dbs = outs_of(q->dB_stride, d.L, d.G, d.N), dcs = outs_of(q->dC_stride, d.L, d.G, d.N);
    const int64_t dt3[4] = {q->ddt_stride[0], q->ddt_stride[1], q->ddt_stride[2], 0};
    const OutS dts = outs_of(dt3, d.L, d.H, 1);
    const cudaError_t e = cudaMemsetAsync(sc.ddtp_exp, 0, scratch_zero_floats(d) * sizeof(float), st);
    if (e != cudaSuccess) {
        set_error("b200_ssd_bwd: cudaMemsetAsync: %s", cudaGetErrorString(e));
        return (int)e;
    }
    if (d.seq.p) {
        if (int rc = bwd_masked<T, true>(q, d, ws, sc, X, Bv, Cv, DO, OUT, dxs, dbs, dcs, st)) return rc;
    } else {
        if (int rc = bwd_masked<T, false>(q, d, ws, sc, X, Bv, Cv, DO, OUT, dxs, dbs, dcs, st)) return rc;
    }
    LAUNCH((dt_bwd_kernel<T>), (size_t)d.batch * d.H * d.nc, d.Q, 0, st, (const T*)p->dt, p->dt_stride[0], p->dt_stride[1],
           p->dt_stride[2], p->A, p->dt_bias, p->dt_softplus, p->dt_min, p->dt_max, d, ws, sc.ddtp_exp, sc.dcs_pos, sc.dcsQ, q->ddt, dts,
           q->dA, q->ddt_bias);
    return 0;
}

}  // namespace ssd
}  // namespace b200

using namespace b200;
using namespace b200::ssd;

static bool dims_ok(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim, int32_t n_groups, int32_t dstate, int32_t chunk) {
    return batch > 0 && seqlen > 0 && nheads > 0 && headdim > 0 && n_groups > 0 && dstate > 0 && chunk > 0 && nheads % n_groups == 0;
}
static Dims dims_of(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim, int32_t n_groups, int32_t dstate, int32_t chunk) {
    Dims d;
    d.batch = batch; d.L = seqlen; d.H = nheads; d.P = headdim; d.G = n_groups; d.N = dstate; d.Q = chunk;
    d.nc = (seqlen + chunk - 1) / chunk;
    d.hpg = nheads / n_groups;
    d.seq = Seq{nullptr, 0, 0};
    return d;
}

extern "C" size_t b200_ssd_workspace_bytes(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim, int32_t n_groups,
                                           int32_t dstate, int32_t chunk_size) {
    if (!dims_ok(batch, seqlen, nheads, headdim, n_groups, dstate, chunk_size)) return 0;
    const Dims d = dims_of(batch, seqlen, nheads, headdim, n_groups, dstate, chunk_size);
    return (2 * ws_dt_floats(d) + ws_state_floats(d) + ws_cb_floats(d)) * sizeof(float);
}

extern "C" size_t b200_ssd_bwd_scratch_bytes(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim, int32_t n_groups,
                                             int32_t dstate, int32_t chunk_size) {
    if (!dims_ok(batch, seqlen, nheads, headdim, n_groups, dstate, chunk_size)) return 0;
    const Dims d = dims_of(batch, seqlen, nheads, headdim, n_groups, dstate, chunk_size);
    return (((scratch_zero_floats(d) + 3) & ~(size_t)3) + ws_state_floats(d) + ws_cb_floats(d)) * sizeof(float);
}

extern "C" int b200_ssd_fwd(const b200_ssd_fwd_params* p, b200_stream_t stream) {
    if (int rc = ssd::validate(p)) return rc;
    B200_REQUIRE(p->out != nullptr, "b200_ssd_fwd: out is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    switch (p->io_dtype) {
        case B200_F32: return fwd_impl<float>(p, st);
        case B200_BF16: return fwd_impl<__nv_bfloat16>(p, st);
        default: return fwd_impl<__half>(p, st);
    }
}

extern "C" int b200_ssd_bwd(const b200_ssd_bwd_params* q, b200_stream_t stream) {
    B200_REQUIRE(q != nullptr, "b200_ssd_bwd: params is NULL");
    if (int rc = ssd::validate(&q->f)) return rc;
    B200_REQUIRE(q->f.out != nullptr, "b200_ssd_bwd: the forward output (f.out) is required");
    B200_REQUIRE(q->dout && q->dx && q->ddt && q->dB && q->dC && q->dA && q->scratch,
                 "b200_ssd_bwd: dout/dx/ddt/dB/dC/dA/scratch must be non-NULL");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(q->scratch) & 15) == 0, "b200_ssd_bwd: scratch must be 16-byte aligned");
    B200_REQUIRE(q->dfinal_states == nullptr || q->final_states != nullptr,
                 "b200_ssd_bwd: dfinal_states needs the forward's final_states");
    B200_REQUIRE(q->dinitial_states == nullptr || q->f.initial_states != nullptr,
                 "b200_ssd_bwd: dinitial_states needs f.initial_states");
    cudaStream_t st = (cudaStream_t)stream;
    switch (q->f.io_dtype) {
        case B200_F32: return bwd_impl<float>(q, st);
        case B200_BF16: return bwd_impl<__nv_bfloat16>(q, st);
        default: return bwd_impl<__half>(q, st);
    }
}

extern "C" int b200_ssd_varlen_states(const b200_ssd_fwd_params* p, const int32_t* cu_seqlens, int32_t nseq, float* states,
                                      b200_stream_t stream) {
    if (int rc = ssd::validate(p)) return rc;
    B200_REQUIRE(p->batch == 1, "b200_ssd_varlen_states: packed sequences need batch == 1 (got %d)", p->batch);
    B200_REQUIRE(cu_seqlens && states, "b200_ssd_varlen_states: cu_seqlens / states must be non-NULL");
    B200_REQUIRE(nseq >= 1 && nseq <= 65535, "b200_ssd_varlen_states: nseq %d must be in [1, 65535]", nseq);
    B200_REQUIRE(p->nheads <= 65535, "b200_ssd_varlen_states: nheads %d > 65535", p->nheads);
    const Dims d = make_dims(*p);
    const Ws ws = make_ws(p->workspace, d);
    const dim3 grid((unsigned)nseq, (unsigned)d.H, (unsigned)((d.P * d.N + NTHR - 1) / NTHR));
    cudaStream_t st = (cudaStream_t)stream;
    switch (p->io_dtype) {
        case B200_F32:
            varlen_states_kernel<float><<<grid, NTHR, 0, st>>>(view4<float>(p->x, p->x_stride), view4<float>(p->B, p->B_stride), d, ws, cu_seqlens, states);
            break;
        case B200_BF16:
            varlen_states_kernel<__nv_bfloat16><<<grid, NTHR, 0, st>>>(view4<__nv_bfloat16>(p->x, p->x_stride), view4<__nv_bfloat16>(p->B, p->B_stride),
                                                                      d, ws, cu_seqlens, states);
            break;
        default:
            varlen_states_kernel<__half><<<grid, NTHR, 0, st>>>(view4<__half>(p->x, p->x_stride), view4<__half>(p->B, p->B_stride), d, ws, cu_seqlens,
                                                               states);
    }
    return check_launch("varlen_states_kernel");
}

extern "C" int b200_rmsnorm_gated_fwd(const float* x, const float* z, const float* w, float* y, float* rstd, int64_t rows, int32_t dim,
                                      float eps, b200_stream_t stream) {
    B200_REQUIRE(x && z && w && y && rstd, "b200_rmsnorm_gated_fwd: NULL pointer");
    B200_REQUIRE(rows > 0 && dim > 0, "b200_rmsnorm_gated_fwd: rows/dim must be positive");
    rmsnorm_gated_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, z, w, y, rstd, rows, dim, eps);
    return check_launch("rmsnorm_gated_fwd_kernel");
}

extern "C" int b200_rmsnorm_gated_bwd(const float* x, const float* z, const float* w, const float* rstd, const float* dy, float* dx,
                                      float* dz, float* dw_partial, int32_t dw_rows, int64_t rows, int32_t dim, b200_stream_t stream) {
    B200_REQUIRE(x && z && w && rstd && dy && dx && dz && dw_partial, "b200_rmsnorm_gated_bwd: NULL pointer");
    B200_REQUIRE(rows > 0 && dim > 0 && dw_rows > 0, "b200_rmsnorm_gated_bwd: rows/dim/dw_rows must be positive");
    B200_REQUIRE(dim <= 12288, "b200_rmsnorm_gated_bwd: dim %d too large", dim);
    const int rpb = (int)((rows + dw_rows - 1) / dw_rows);
    rmsnorm_gated_bwd_kernel<<<(unsigned)dw_rows, 256, dim * sizeof(float), (cudaStream_t)stream>>>(x, z, w, rstd, dy, dx, dz, dw_partial,
                                                                                                  rows, dim, rpb);
    return check_launch("rmsnorm_gated_bwd_kernel");
}
