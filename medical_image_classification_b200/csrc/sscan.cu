// sscan.cu -- Mamba-1 selective scan, forward and backward, for sm_100a.
//
// Replaces selective_scan_cuda.fwd/.bwd (reference CrossMamba/FusionMamba/selective_scan/
// selective_scan_fwd_kernel.cuh:67-303, selective_scan_bwd_kernel.cuh:75-489).  Not a port: the
// reference maps one CTA to one (batch, channel) row and runs a CUB block scan per state; here
//
//   * the unit of work ("task") is ONE WARP: 16 consecutive channels of one (batch, group), all 16 states.
//     Lane = (state quad sq = lane >> 3, row pair i = lane & 7): the lane owns rows i and i + 8 -- carried
//     as the two halves of packed f32x2 registers (FFMA2/FMUL2: one issue slot, two rows) -- and states
//     4 sq .. 4 sq + 3.  The time recurrence is an in-register FFMA chain: no block scan, every
//     exp(delta * A) is evaluated exactly once, and warps never wait for one another (no block barrier
//     anywhere in the kernels; a CTA is just four independent tasks);
//   * u / delta / dout tiles (16 rows x 8 steps), the group's B / C tile (16 states x 8 steps) and the
//     8-step state checkpoint stream in through a per-warp double-buffered cp.async pipeline (16-byte
//     copies when the tensors allow it), XOR-swizzled / padded so every shared-memory read below is
//     conflict free;
//   * softplus(delta + bias) (and its derivative) is evaluated once per element: each lane does the 4
//     elements (2 rows x 2 steps) it owns and the warp all-gathers them through a 2 KB exchange tile;
//   * reductions over states (y, d delta, d u) are 4 in-register FMAs + a 4-lane reduce-scatter, reductions
//     over channels (dB, dC) are an in-register row-pair sum + an 8-lane reduce-scatter that leaves lane i
//     with the total of step i: one fully used fp32 RED per (state, chunk, quantity);
//   * a group can be scanned in reverse time (rev_mask) and groups can share u / dout rows (u_group_div,
//     dout_group_div): that is all the SS2D cross-scan / cross-merge needs (MedMamba.py:393-395, 420-424),
//     the flipped copies never exist.  Register arrays and the exchange tiles are indexed by SCAN step; the
//     direction only changes (warp-uniform, run-time) shared-memory addresses, so there is one code body;
//   * backward = recompute: the forward stores the 16-float state entering every 8-step chunk, the backward
//     walks chunks last -> first, re-derives the states of one chunk in registers and runs the adjoint
//     recurrence on them.
//
// Binding pipes (DESIGN.md): forward = MUFU.EX2 (16 per element) with issue close behind, backward = issue.
#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no libcuda link)

#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "common.cuh"

namespace b200 {

constexpr int NS = 16;   // states per task
constexpr int SPT = 4;   // states per thread
constexpr int TR = B200_SSCAN_ROWS_PER_TASK;  // rows per task
constexpr int TC = 8;    // steps per chunk == checkpoint interval
constexpr int WPB = 1;   // warps (independent tasks) per CTA
constexpr int EXS = 24;  // exchange tile: words per column (16 used; 24 keeps the STS.64 conflict free)
constexpr int BCS = 40;  // B/C tile: words per state quad (4 states x 8 steps + 8 pad)
constexpr int CKS = 80;  // checkpoint tile: words per state quad (4 states x 8 row pairs x 2 + 16 pad)
constexpr int RDS = 144; // state-reduction tile: words per state quad (8 columns x 8 row pairs x 2 + 16 pad)
constexpr float kLn2 = 0.6931471805599453f;
static_assert(TR == 16, "lane mapping assumes 16 rows per task");

// ---- cp.async (LDGSTS) -----------------------------------------------------------------------
__device__ __forceinline__ void cp_async4(float* smem, const float* gmem, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int n = pred ? 4 : 0;  // src-size 0 => the destination bytes are zero-filled
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(s), "l"(gmem), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async16(float* smem, const float* gmem, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int n = pred ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async16_ca(float* smem, const float* gmem, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int n = pred ? 16 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }


// ---- TMA (cp.async.bulk.tensor) + mbarrier: the u / delta / dout tiles of the aligned fp32 path -------------
// One 16 x 8 box per tensor and chunk, issued by lane 0, completion counted in bytes on a per-stage mbarrier.
// SWIZZLE_32B is exactly raw_pos() (16-byte half of a 32-byte row XOR bit 2 of the row index), rows / positions
// outside the tensor are zero-filled by the copy engine, and none of this traffic touches the LSU wavefront pipe.
struct RowMaps {
    CUtensorMap u, delta, dout;   // 4-D: (L, rows per group, groups, batch)
};
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(float* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(dst)),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
// generic-proxy writes / reads of a tile must be ordered before the async proxy (TMA) overwrites it
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
constexpr unsigned ROW_TILE_BYTES = TR * TC * sizeof(float);

struct Task {
    int b, g, r0, nrows, rpg, d0;  // d0 = first channel of the task
    bool rev;
};

__host__ __device__ __forceinline__ int tiles_per_group(int rpg) { return (rpg + TR - 1) / TR; }

__device__ __forceinline__ Task decode_task(const b200_sscan_fwd_params& p, long long task) {
    Task t;
    t.rpg = p.dim / p.n_groups;
    const int tiles = tiles_per_group(t.rpg);
    const int rt = (int)(task % tiles);
    const int bg = (int)(task / tiles);
    t.g = bg % p.n_groups;
    t.b = bg / p.n_groups;
    t.r0 = rt * TR;
    t.nrows = min(TR, t.rpg - t.r0);
    t.d0 = t.g * t.rpg + t.r0;
    t.rev = (p.rev_mask >> t.g) & 1u;
    return t;
}

// ---- shared-memory tile layouts -------------------------------------------------------------------
// raw activation tile: 16 rows x 8 steps, pitch 8, the two 16-byte halves of a row swapped on rows 4-7 / 12-15
__device__ __forceinline__ int raw_pos(int row, int c) { return row * TC + (c ^ (((row >> 2) & 1) << 2)); }
// B / C tile: [state quad][state in quad][8 steps], quads 40 words apart
__device__ __forceinline__ int bc_pos(int n, int c) { return (n >> 2) * BCS + (n & 3) * TC + c; }

// One 16-byte cp.async per lane and chunk moves a whole [16 rows or states][8 steps] fp32 tile.  Everything that
// does not depend on the chunk (source row pointer, shared-memory slot, row validity) is computed once per task.
struct Stager {
    const float* src;   // this lane's row at sequence position 0
    unsigned dst;       // shared address of the lane's 16-byte slot in stage 0
    bool ok;
};
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16_s(unsigned dst, const float* src, bool pred, bool ca) {
    const int n = pred ? 16 : 0;
    if (ca) asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
    else asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ Stager make_row_stager(float* tile, const float* base, int64_t row_stride, int nrows, int lane) {
    const int row = lane >> 1, c = (lane & 1) * 4;
    Stager s;
    s.ok = row < nrows;
    s.src = base + (s.ok ? (size_t)row * row_stride : 0);
    s.dst = smem_u32(tile + raw_pos(row, c));
    return s;
}
__device__ __forceinline__ Stager make_bc_stager(float* tile, const float* base, int64_t state_stride, int N, int lane) {
    const int n = lane >> 1, c = (lane & 1) * 4;
    Stager s;
    s.ok = n < N;
    s.src = base + (s.ok ? (size_t)n * state_stride : 0);
    s.dst = smem_u32(tile + bc_pos(n, c));
    return s;
}
// l = l_lo + this lane's first column; the 4 positions are all inside or all outside [0, L) (L % 4 == 0)
__device__ __forceinline__ void stage16(const Stager& s, unsigned stage_off, int l, int L, bool ca) {
    const bool ok = s.ok && (unsigned)l < (unsigned)L;
    cp_async16_s(s.dst + stage_off, ok ? s.src + l : s.src, ok, ca);
}

// ---- 16-bit I/O: the same double-buffered pipeline with one 8-byte cp.async (4 elements) per lane and tile.  Tiles stay
// 16-bit in shared memory, [16 rows or states][8 steps] with a 16-byte pitch: the activation tile in the first half of its
// fp32 slot, the B / C tiles in the second halves of slots 0 / 1 (converted to the fp32 B / C tiles once per chunk).
struct Stager16 {
    const char* src;
    unsigned dst;
    bool ok;
};
template <typename T>
__device__ __forceinline__ Stager16 make_stager16(float* slot, int elem_off, const T* base, int64_t stride, int nvalid, int lane) {
    const int r = lane >> 1, c = (lane & 1) * 4;
    Stager16 s;
    s.ok = r < nvalid;
    s.src = reinterpret_cast<const char*>(base + (s.ok ? (size_t)r * stride : 0));
    s.dst = smem_u32(reinterpret_cast<T*>(slot) + elem_off + r * TC + c);
    return s;
}
__device__ __forceinline__ void stage8(const Stager16& s, unsigned stage_off, int l, int L) {
    const bool ok = s.ok && (unsigned)l < (unsigned)L;
    const int n = ok ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(s.dst + stage_off), "l"(ok ? s.src + 2 * (size_t)l : s.src), "r"(n)
                 : "memory");
}
template <typename T> __device__ __forceinline__ float2 unpack2(unsigned w) {
    if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
    } else {
        return __half22float2(*reinterpret_cast<const __half2*>(&w));
    }
}
// rows i and i + 8, columns c0 and c0 + 1 of a staged 16-bit activation tile
template <typename T> __device__ __forceinline__ void read_rows16(const float* slot, int i, int sq, float (&a)[2], float (&b)[2]) {
    const unsigned* w = reinterpret_cast<const unsigned*>(slot);
    const float2 va = unpack2<T>(w[i * 4 + sq]), vb = unpack2<T>(w[(i + 8) * 4 + sq]);
    a[0] = va.x; a[1] = va.y; b[0] = vb.x; b[1] = vb.y;
}
// staged 16-bit B or C tile (second half of a raw slot) -> fp32 tile in the bc_pos layout; 4 elements per lane
template <typename T> __device__ __forceinline__ void convert_bc16(float* tile, const float* slot, int lane) {
    const int n = lane >> 1, c = (lane & 1) * 4;
    const uint2 w = *reinterpret_cast<const uint2*>(reinterpret_cast<const T*>(slot) + TR * TC + n * TC + c);
    const float2 lo = unpack2<T>(w.x), hi = unpack2<T>(w.y);
    *reinterpret_cast<float4*>(tile + bc_pos(n, c)) = make_float4(lo.x, lo.y, hi.x, hi.y);
}

// Element-wise fallbacks (L % 4 != 0 or unaligned views): column c <-> sequence position l_lo + c; out-of-range -> 0.
__device__ __forceinline__ void stage_rows_slow(float* tile, const float* base, int64_t row_stride, int nrows, int l_lo, int L, int lane) {
#pragma unroll 1
    for (int k = 0; k < TR * TC / 32; ++k) {
        const int idx = k * 32 + lane;
        const int row = idx >> 3, c = idx & 7;
        const int l = l_lo + c;
        const bool ok = row < nrows && l >= 0 && l < L;
        cp_async4(tile + raw_pos(row, c), ok ? base + (size_t)row * row_stride + l : base, ok);
    }
}
__device__ __forceinline__ void stage_bc_slow(float* tile, const float* base, int64_t state_stride, int N, int l_lo, int L, int lane) {
#pragma unroll 1
    for (int k = 0; k < NS * TC / 32; ++k) {
        const int idx = k * 32 + lane;
        const int n = idx >> 3, c = idx & 7;
        const int l = l_lo + c;
        const bool ok = n < N && l >= 0 && l < L;
        cp_async4(tile + bc_pos(n, c), ok ? base + (size_t)n * state_stride + l : base, ok);
    }
}

// Synchronous variants for 16-bit I/O (converted on the fly).
template <typename T>
__device__ __forceinline__ void fill_bc_sync(float* tile, const T* base, int64_t state_stride, int N, int l_lo, int L, int lane) {
#pragma unroll
    for (int k = 0; k < NS * TC / 32; ++k) {
        const int idx = k * 32 + lane;
        const int n = idx >> 3, c = idx & 7;
        const int l = l_lo + c;
        const bool ok = n < N && l >= 0 && l < L;
        tile[bc_pos(n, c)] = ok ? to_f32<T>(__ldg(base + (size_t)n * state_stride + l)) : 0.f;
    }
}

// One chunk of checkpoints (256 floats, record layout: ckpt_state_pos in common.cuh) -> padded tile [n][row pair][2].
__device__ __forceinline__ void stage_ckpt(float* tile, const float* src, int lane) {
#pragma unroll
    for (int k0 = 0; k0 < NS * TR / 4; k0 += 32) {
        const int k = k0 + lane;
        const int n = k >> 2, part = k & 3;
        cp_async16(tile + (n >> 2) * CKS + (n & 3) * 16 + part * 4, src + ckpt_state_pos(n) + part * 4, true);
    }
}

template <typename T>
__device__ __forceinline__ bool can_vectorize(const void* p, int64_t row_stride, int64_t batch_stride, int64_t group_stride,
                                              int L) {
    return (L & 3) == 0 && (row_stride & 3) == 0 && (batch_stride & 3) == 0 && (group_stride & 3) == 0 &&
           (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(T) - 1)) == 0;   // 4 elements per cp.async: 16 bytes fp32, 8 bytes 16-bit
}

// two adjacent sequence positions of one row
template <typename T> __device__ __forceinline__ void store_pair(T* p, float a, float b, bool ok0, bool ok1, bool vec) {
    if (vec && ok0 && ok1) {
        if constexpr (sizeof(T) == 4) {
            __stcs(reinterpret_cast<float2*>(p), make_float2(a, b));
        } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
            const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
            __stcs(reinterpret_cast<unsigned int*>(p), *reinterpret_cast<const unsigned int*>(&v));
        } else {
            const __half2 v = __floats2half2_rn(a, b);
            __stcs(reinterpret_cast<unsigned int*>(p), *reinterpret_cast<const unsigned int*>(&v));
        }
    } else {
        if (ok0) stg_stream(p, a);
        if (ok1) stg_stream(p + 1, b);
    }
}
template <typename T> __device__ __forceinline__ bool pair_vec_ok(const void* p, int64_t row_stride, int64_t batch_stride, int L) {
    return (L & 1) == 0 && (row_stride & 1) == 0 && (batch_stride & 1) == 0 && (reinterpret_cast<uintptr_t>(p) & (2 * sizeof(T) - 1)) == 0;
}

__device__ __forceinline__ float2 ex2_2(float2 e) { return make_float2(ex2(e.x), ex2(e.y)); }

// ---- warp reductions -----------------------------------------------------------------------------
// Reduce-scatter of 8 per-lane values over the 8 lanes that share a state quad (lane bits 0-2): lane i ends
// with the 8-lane total of v[i].  7 shuffles instead of 24.
__device__ __forceinline__ float rs8_rows(const float (&v)[8], int lane) {
    float h4[4], h2[2];
    const bool u4 = lane & 4, u2 = lane & 2, u1 = lane & 1;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float keep = u4 ? v[k + 4] : v[k], send = u4 ? v[k] : v[k + 4];
        h4[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float keep = u2 ? h4[k + 2] : h4[k], send = u2 ? h4[k] : h4[k + 2];
        h2[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    const float keep = u1 ? h2[1] : h2[0], send = u1 ? h2[0] : h2[1];
    return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

// One state's 8 steps of B or C in SCAN order (v[s] <-> memory column rev ? 7 - s : s).  The branch is warp-uniform.
__device__ __forceinline__ void load8_steps(const float* p, bool rev, float (&v)[TC]) {
    if (!rev) {
        const float4 lo = *reinterpret_cast<const float4*>(p), hi = *reinterpret_cast<const float4*>(p + 4);
        v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    } else {
#pragma unroll
        for (int s = 0; s < TC; ++s) v[s] = p[TC - 1 - s];
    }
}

// Sum 8 per-lane row-pair values over the 4 state quads (lane bits 3-4) through a 2.3 KB shared-memory tile: the
// lane ends with the totals of the two scan steps s0, s1 that correspond to the two memory columns (2 sq, 2 sq + 1)
// whose elements it owns in the prologue / epilogue.  8 STS.64 + 8 LDS.64 + 6 packed adds (a shuffle reduce-scatter costs ~100 issue slots).
// The tile layout [quad][column][row pair] is padded (RDS) and XOR-skewed so both phases are conflict free.
__device__ __forceinline__ int rd_pos(int quad, int cc, int i) { return quad * RDS + ((cc * 16 + 2 * i) ^ (((cc >> 1) & 1) << 4)); }
__device__ __forceinline__ void reduce_states(float* tile, const float2 (&v)[8], int lane, int s0, int s1, float2& r0, float2& r1) {
    const int sq = lane >> 3, i = lane & 7;
#pragma unroll
    for (int s = 0; s < 8; ++s) *reinterpret_cast<float2*>(tile + rd_pos(sq, s, i)) = v[s];
    __syncwarp();
    r0 = *reinterpret_cast<const float2*>(tile + rd_pos(0, s0, i));   // s0 / s1: the scan steps of this lane's two columns
    r1 = *reinterpret_cast<const float2*>(tile + rd_pos(0, s1, i));
#pragma unroll
    for (int qd = 1; qd < 4; ++qd) {
        r0 = __fadd2_rn(r0, *reinterpret_cast<const float2*>(tile + rd_pos(qd, s0, i)));
        r1 = __fadd2_rn(r1, *reinterpret_cast<const float2*>(tile + rd_pos(qd, s1, i)));
    }
}

// ----------------------------------------------------------------------------------------------
// forward
// ----------------------------------------------------------------------------------------------
struct FwdWarpSmem {
    float raw[2][2][TR * TC];      // [stage][u, delta]
    float bc[2][2][4 * BCS];       // [stage][B, C]
    float ex[2][TC * EXS];         // delta' | delta' * u, [column][row pair][2]
    float rd[4 * RDS];             // reduction over the state quads
    uint64_t bar[2];               // TMA completion, one per stage
};

template <typename T, bool HAS_Z, bool TMA>
__device__ __forceinline__ void sscan_fwd_body(const b200_sscan_fwd_params& p, const RowMaps& tm, const Task& t,
                                               long long task, FwdWarpSmem& sm, int lane) {
    constexpr bool ASYNC = sizeof(T) == 4;
    const int sq = lane >> 3, i = lane & 7;
    const int L = p.seqlen, N = p.dstate;
    const int c0 = 2 * sq;  // this lane's two columns in the prologue / epilogue
    const bool okA = i < t.nrows, okB = i + 8 < t.nrows;
    const int dA_ = t.d0 + i, dB_ = t.d0 + i + 8;

    float2 A2[SPT], x[SPT];
#pragma unroll
    for (int j = 0; j < SPT; ++j) {
        const int n = sq * SPT + j;
        A2[j].x = (okA && n < N) ? __ldg(p.A + (size_t)dA_ * N + n) * kLog2e : 0.f;
        A2[j].y = (okB && n < N) ? __ldg(p.A + (size_t)dB_ * N + n) * kLog2e : 0.f;
        x[j] = make_float2(0.f, 0.f);
    }
    const float biasA = (p.delta_bias && okA) ? __ldg(p.delta_bias + dA_) : 0.f;
    const float biasB = (p.delta_bias && okB) ? __ldg(p.delta_bias + dB_) : 0.f;
    const float DA = (p.D && okA) ? __ldg(p.D + dA_) : 0.f;
    const float DB = (p.D && okB) ? __ldg(p.D + dB_) : 0.f;
    const bool softplus = p.delta_softplus != 0;

    const T* u_base = (const T*)p.u + (size_t)t.b * p.u_batch_stride + (size_t)(t.g / p.u_group_div) * p.u_group_stride +
                      (size_t)t.r0 * p.u_row_stride;
    const T* d_base = (const T*)p.delta + (size_t)t.b * p.delta_batch_stride + (size_t)t.g * p.delta_group_stride +
                      (size_t)t.r0 * p.delta_row_stride;
    T* o_base = (T*)p.out + (size_t)t.b * p.out_batch_stride + (size_t)t.d0 * p.out_row_stride;
    const T* z_base = HAS_Z ? (const T*)p.z + (size_t)t.b * p.z_batch_stride + (size_t)t.d0 * p.z_row_stride : nullptr;
    const T* B_base = (const T*)p.B + (size_t)t.b * p.B_batch_stride + (size_t)t.g * p.B_group_stride;
    const T* C_base = (const T*)p.C + (size_t)t.b * p.C_batch_stride + (size_t)t.g * p.C_group_stride;
    const bool vec_u = can_vectorize<T>(p.u, p.u_row_stride, p.u_batch_stride, p.u_group_stride, L);
    const bool vec_d = can_vectorize<T>(p.delta, p.delta_row_stride, p.delta_batch_stride, p.delta_group_stride, L);
    const bool vec_B = can_vectorize<T>(p.B, p.B_state_stride, p.B_batch_stride, p.B_group_stride, L);
    const bool vec_C = can_vectorize<T>(p.C, p.C_state_stride, p.C_batch_stride, p.C_group_stride, L);
    const bool vec_o = pair_vec_ok<T>(p.out, p.out_row_stride, p.out_batch_stride, L);

    const int nck = (L + TC - 1) / TC;
    float* ck = p.ckpt ? p.ckpt + (size_t)task * (size_t)(nck - 1) * NS * TR : nullptr;

    const bool rev = t.rev;
    const int st0 = rev ? TC - 1 - c0 : c0, st1 = rev ? TC - 2 - c0 : c0 + 1;  // scan steps of this lane's two columns
    auto l_lo_of = [&](int c) { return rev ? L - (c + 1) * TC : c * TC; };
    const bool fast = vec_u && vec_d && vec_B && vec_C;
    constexpr bool tma = TMA;   // host guarantees `fast` whenever it picks the TMA instantiation
    const Stager su = make_row_stager(sm.raw[0][0], (const float*)u_base, p.u_row_stride, t.nrows, lane);
    const Stager sd = make_row_stager(sm.raw[0][1], (const float*)d_base, p.delta_row_stride, t.nrows, lane);
    const Stager sB = make_bc_stager(sm.bc[0][0], (const float*)B_base, p.B_state_stride, N, lane);
    const Stager sC = make_bc_stager(sm.bc[0][1], (const float*)C_base, p.C_state_stride, N, lane);
    Stager16 hu, hd, hB, hC;
    if constexpr (!ASYNC) {
        hu = make_stager16<T>(sm.raw[0][0], 0, u_base, p.u_row_stride, t.nrows, lane);
        hd = make_stager16<T>(sm.raw[0][1], 0, d_base, p.delta_row_stride, t.nrows, lane);
        hB = make_stager16<T>(sm.raw[0][0], TR * TC, B_base, p.B_state_stride, N, lane);
        hC = make_stager16<T>(sm.raw[0][1], TR * TC, C_base, p.C_state_stride, N, lane);
    }
    const int lc = (lane & 1) * 4;
    auto prefetch = [&](int c) {
        if (ASYNC || fast) {
            if (c < nck) {
                const int buf = c & 1, l_lo = l_lo_of(c);
                if constexpr (!ASYNC) {
                    const int l = l_lo + lc;
                    const unsigned off = buf * (unsigned)sizeof(sm.raw[0]);
                    stage8(hu, off, l, L);
                    stage8(hd, off, l, L);
                    stage8(hB, off, l, L);
                    stage8(hC, off, l, L);
                } else if (fast) {
                    const int l = l_lo + lc;
                    if (tma) {
                        if (lane == 0) {
                            mbar_expect_tx(&sm.bar[buf], 2 * ROW_TILE_BYTES);
                            tma_load_4d(sm.raw[buf][0], &tm.u, l_lo, t.r0, t.g / p.u_group_div, t.b, &sm.bar[buf]);
                            tma_load_4d(sm.raw[buf][1], &tm.delta, l_lo, t.r0, t.g, t.b, &sm.bar[buf]);
                        }
                    } else {
                        stage16(su, buf * (unsigned)sizeof(sm.raw[0]), l, L, false);
                        stage16(sd, buf * (unsigned)sizeof(sm.raw[0]), l, L, false);
                    }
                    stage16(sB, buf * (unsigned)sizeof(sm.bc[0]), l, L, true);
                    stage16(sC, buf * (unsigned)sizeof(sm.bc[0]), l, L, true);
                } else {
                    stage_rows_slow(sm.raw[buf][0], (const float*)u_base, p.u_row_stride, t.nrows, l_lo, L, lane);
                    stage_rows_slow(sm.raw[buf][1], (const float*)d_base, p.delta_row_stride, t.nrows, l_lo, L, lane);
                    stage_bc_slow(sm.bc[buf][0], (const float*)B_base, p.B_state_stride, N, l_lo, L, lane);
                    stage_bc_slow(sm.bc[buf][1], (const float*)C_base, p.C_state_stride, N, l_lo, L, lane);
                }
            }
            cp_async_commit();  // (possibly empty) group: keeps the wait_group arithmetic uniform
        }
    };
    if (tma) {
        if (lane == 0) {
            mbar_init(&sm.bar[0], 1);
            mbar_init(&sm.bar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }
    // software pipeline with ONE prefetch call site (code size): iterations -2 and -1 only prefetch
    for (int c = -2; c < nck; ++c) {
        if (c < 0) {
            prefetch(c + 2);
            continue;
        }
        const int buf = c & 1;
        const int l_lo = l_lo_of(c);
        const int la = l_lo + c0;  // sequence position of this lane's first column
        const bool v0 = la >= 0 && la < L, v1 = la + 1 >= 0 && la + 1 < L;
        float uA[2], uB[2], dlA[2], dlB[2];
        if (ASYNC) {
            cp_async_wait<1>();
            if (tma) mbar_wait(&sm.bar[buf], (c >> 1) & 1);   // the (c >> 1)-th use of this stage
            __syncwarp();
            const float2 ua = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i, c0)]);
            const float2 ub = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i + 8, c0)]);
            const float2 da = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i, c0)]);
            const float2 db = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i + 8, c0)]);
            uA[0] = ua.x; uA[1] = ua.y; uB[0] = ub.x; uB[1] = ub.y;
            dlA[0] = da.x; dlA[1] = da.y; dlB[0] = db.x; dlB[1] = db.y;
        } else if (fast) {
            cp_async_wait<1>();
            __syncwarp();
            read_rows16<T>(sm.raw[buf][0], i, sq, uA, uB);
            read_rows16<T>(sm.raw[buf][1], i, sq, dlA, dlB);
            convert_bc16<T>(sm.bc[buf][0], sm.raw[buf][0], lane);
            convert_bc16<T>(sm.bc[buf][1], sm.raw[buf][1], lane);
        } else {
            fill_bc_sync<T>(sm.bc[buf][0], B_base, p.B_state_stride, N, l_lo, L, lane);
            fill_bc_sync<T>(sm.bc[buf][1], C_base, p.C_state_stride, N, l_lo, L, lane);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const bool v = e ? v1 : v0;
                uA[e] = (okA && v) ? ldg_stream(u_base + (size_t)i * p.u_row_stride + la + e) : 0.f;
                uB[e] = (okB && v) ? ldg_stream(u_base + (size_t)(i + 8) * p.u_row_stride + la + e) : 0.f;
                dlA[e] = (okA && v) ? ldg_stream(d_base + (size_t)i * p.delta_row_stride + la + e) : 0.f;
                dlB[e] = (okB && v) ? ldg_stream(d_base + (size_t)(i + 8) * p.delta_row_stride + la + e) : 0.f;
            }
        }
        // ---- prologue: delta' = softplus(delta + bias) once per element; q = delta' * u ----
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool v = e ? v1 : v0;
            float a = dlA[e] + biasA, b = dlB[e] + biasB;
            if (softplus) { a = softplus_sigmoid(a).sp; b = softplus_sigmoid(b).sp; }
            dlA[e] = (okA && v) ? a : 0.f;  // out-of-range steps / rows become the identity: decay 1, input 0
            dlB[e] = (okB && v) ? b : 0.f;
            const int st = e ? st1 : st0;   // the exchange tile is indexed by scan step
            *reinterpret_cast<float2*>(&sm.ex[0][st * EXS + 2 * i]) = make_float2(dlA[e], dlB[e]);
            *reinterpret_cast<float2*>(&sm.ex[1][st * EXS + 2 * i]) = make_float2(dlA[e] * uA[e], dlB[e] * uB[e]);
        }
        __syncwarp();
        float2 dl2[TC], q2[TC], y2[TC];   // indexed by scan step
#pragma unroll
        for (int cc = 0; cc < TC; ++cc) {
            dl2[cc] = *reinterpret_cast<const float2*>(&sm.ex[0][cc * EXS + 2 * i]);
            q2[cc] = *reinterpret_cast<const float2*>(&sm.ex[1][cc * EXS + 2 * i]);
            y2[cc] = make_float2(0.f, 0.f);
        }
        // ---- recurrence: this lane's 4 states, one after the other, 2 rows per packed instruction ----
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
            const int n = sq * SPT + j;
            if (ck != nullptr && c > 0) *reinterpret_cast<float2*>(ck + (size_t)(c - 1) * NS * TR + ckpt_state_pos(n) + 2 * i) = x[j];
            float Bv[TC], Cv[TC];
            load8_steps(&sm.bc[buf][0][sq * BCS + j * TC], rev, Bv);
            load8_steps(&sm.bc[buf][1][sq * BCS + j * TC], rev, Cv);
            float2 xs = x[j];
#pragma unroll
            for (int s = 0; s < TC; ++s) {
                const int cc = s;
                const float2 a = ex2_2(__fmul2_rn(dl2[cc], A2[j]));
                const float2 qB = make_float2(q2[cc].x * Bv[cc], q2[cc].y * Bv[cc]);
                xs = __ffma2_rn(a, xs, qB);
                y2[cc].x = fmaf(Cv[cc], xs.x, y2[cc].x);
                y2[cc].y = fmaf(Cv[cc], xs.y, y2[cc].y);
            }
            x[j] = xs;
        }
        // ---- out = sum over states (4 lanes) + D u (* silu(z)), written at its memory position ----
        float2 r0, r1;
        reduce_states(sm.rd, y2, lane, st0, st1, r0, r1);
        float oA[2] = {fmaf(DA, uA[0], r0.x), fmaf(DA, uA[1], r1.x)};
        float oB[2] = {fmaf(DB, uB[0], r0.y), fmaf(DB, uB[1], r1.y)};
        if (HAS_Z) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const bool v = e ? v1 : v0;
                if (okA && v) { const float zz = ldg_stream(z_base + (size_t)i * p.z_row_stride + la + e); oA[e] *= zz * sigmoidf_(zz); }
                if (okB && v) { const float zz = ldg_stream(z_base + (size_t)(i + 8) * p.z_row_stride + la + e); oB[e] *= zz * sigmoidf_(zz); }
            }
        }
        store_pair<T>(o_base + (size_t)i * p.out_row_stride + la, oA[0], oA[1], okA && v0, okA && v1, vec_o);
        store_pair<T>(o_base + (size_t)(i + 8) * p.out_row_stride + la, oB[0], oB[1], okB && v0, okB && v1, vec_o);
        if (tma) fence_proxy_async();
        __syncwarp();  // every lane is done with this chunk's tiles
        prefetch(c + 2);
    }
    if (ASYNC || fast) cp_async_wait<0>();
    if (p.last_state != nullptr) {
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
            const int n = sq * SPT + j;
            if (n < N) {
                if (okA) p.last_state[((size_t)t.b * p.dim + dA_) * N + n] = x[j].x;
                if (okB) p.last_state[((size_t)t.b * p.dim + dB_) * N + n] = x[j].y;
            }
        }
    }
}

template <typename T, bool HAS_Z, bool TMA>
__global__ void __launch_bounds__(WPB * 32, 16) sscan_fwd_kernel(const __grid_constant__ b200_sscan_fwd_params p, const __grid_constant__ RowMaps tm) {
    __shared__ __align__(1024) FwdWarpSmem sm;
    static_assert(WPB == 1, "one warp-task per CTA");
    const int lane = threadIdx.x;
    const long long task = blockIdx.x;
    const Task t = decode_task(p, task);
    sscan_fwd_body<T, HAS_Z, TMA>(p, tm, t, task, sm, lane);
}

// ----------------------------------------------------------------------------------------------
// backward
// ----------------------------------------------------------------------------------------------
struct BwdWarpSmem {
    float raw[2][3][TR * TC];   // [stage][u, delta -> sigmoid(delta + bias), dout]
    float bc[2][2][4 * BCS];    // [stage][B, C]
    float ck[2][4 * CKS];       // state entering the chunk
    float ex[3][TC * EXS];      // delta' | delta' * u | gated dout, [column][row pair][2]
    float rd[4 * RDS];          // reduction over the state quads
    float2 A2[SPT][32];         // per-lane constants / accumulators that would not fit in registers:
    float2 dA[SPT][32];         // A * log2(e), the running dA and the adjoint carry of the lane's 4 states x 2 rows
    float2 h[SPT][32];
    uint64_t bar[2];            // TMA completion, one per stage
};

template <typename T, bool HAS_Z, bool TMA>
__device__ __forceinline__ void sscan_bwd_body(const b200_sscan_bwd_params& q, const RowMaps& tm, const Task& t,
                                               long long task, BwdWarpSmem& sm, int lane) {
    const b200_sscan_fwd_params& p = q.f;
    constexpr bool ASYNC = sizeof(T) == 4;
    const int sq = lane >> 3, i = lane & 7;
    const int L = p.seqlen, N = p.dstate;
    const int c0 = 2 * sq;
    const bool okA = i < t.nrows, okB = i + 8 < t.nrows;
    const int dA_ = t.d0 + i, dB_ = t.d0 + i + 8;

#pragma unroll
    for (int j = 0; j < SPT; ++j) {
        const int n = sq * SPT + j;
        float2 a2;
        a2.x = (okA && n < N) ? __ldg(p.A + (size_t)dA_ * N + n) * kLog2e : 0.f;
        a2.y = (okB && n < N) ? __ldg(p.A + (size_t)dB_ * N + n) * kLog2e : 0.f;
        sm.A2[j][lane] = a2;   // private to this lane: no synchronisation needed
        sm.dA[j][lane] = make_float2(0.f, 0.f);
        sm.h[j][lane] = make_float2(0.f, 0.f);
    }
    const float biasA = (p.delta_bias && okA) ? __ldg(p.delta_bias + dA_) : 0.f;
    const float biasB = (p.delta_bias && okB) ? __ldg(p.delta_bias + dB_) : 0.f;
    const float DA = (p.D && okA) ? __ldg(p.D + dA_) : 0.f;
    const float DB = (p.D && okB) ? __ldg(p.D + dB_) : 0.f;
    const bool softplus = p.delta_softplus != 0;
    float dD_A = 0.f, dD_B = 0.f, dbias_A = 0.f, dbias_B = 0.f;  // this lane's share (its two columns of every chunk)

    const T* u_base = (const T*)p.u + (size_t)t.b * p.u_batch_stride + (size_t)(t.g / p.u_group_div) * p.u_group_stride +
                      (size_t)t.r0 * p.u_row_stride;
    const T* d_base = (const T*)p.delta + (size_t)t.b * p.delta_batch_stride + (size_t)t.g * p.delta_group_stride +
                      (size_t)t.r0 * p.delta_row_stride;
    const T* g_base = (const T*)q.dout + (size_t)t.b * q.dout_batch_stride +
                      (size_t)(t.g / (int)q.dout_group_div) * q.dout_group_stride + (size_t)t.r0 * q.dout_row_stride;
    const T* z_base = HAS_Z ? (const T*)p.z + (size_t)t.b * p.z_batch_stride + (size_t)t.d0 * p.z_row_stride : nullptr;
    T* du_base = (T*)q.du + (size_t)t.b * q.du_batch_stride + (size_t)t.d0 * q.du_row_stride;
    T* dd_base = (T*)q.ddelta + (size_t)t.b * q.ddelta_batch_stride + (size_t)t.g * q.ddelta_group_stride +
                 (size_t)t.r0 * q.ddelta_row_stride;
    T* dz_base = HAS_Z ? (T*)q.dz + (size_t)t.b * q.dz_batch_stride + (size_t)t.d0 * q.dz_row_stride : nullptr;
    const T* B_base = (const T*)p.B + (size_t)t.b * p.B_batch_stride + (size_t)t.g * p.B_group_stride;
    const T* C_base = (const T*)p.C + (size_t)t.b * p.C_batch_stride + (size_t)t.g * p.C_group_stride;
    float* dB_base = q.dB + (size_t)t.b * q.dB_batch_stride + (size_t)t.g * q.dB_group_stride;
    float* dC_base = q.dC + (size_t)t.b * q.dC_batch_stride + (size_t)t.g * q.dC_group_stride;
    const int dBs = (int)q.dB_state_stride, dCs = (int)q.dC_state_stride;   // N * stride < 2^31 (checked on the host)
    const bool vec_u = can_vectorize<T>(p.u, p.u_row_stride, p.u_batch_stride, p.u_group_stride, L);
    const bool vec_d = can_vectorize<T>(p.delta, p.delta_row_stride, p.delta_batch_stride, p.delta_group_stride, L);
    const bool vec_g = can_vectorize<T>(q.dout, q.dout_row_stride, q.dout_batch_stride, q.dout_group_stride, L);
    const bool vec_B = can_vectorize<T>(p.B, p.B_state_stride, p.B_batch_stride, p.B_group_stride, L);
    const bool vec_C = can_vectorize<T>(p.C, p.C_state_stride, p.C_batch_stride, p.C_group_stride, L);
    const bool vec_du = pair_vec_ok<T>(q.du, q.du_row_stride, q.du_batch_stride, L);
    const bool vec_dd = pair_vec_ok<T>(q.ddelta, q.ddelta_row_stride, q.ddelta_batch_stride, L) && (q.ddelta_group_stride & 1) == 0;
    const bool vec_dz = HAS_Z && pair_vec_ok<T>(q.dz, q.dz_row_stride, q.dz_batch_stride, L);

    const int nck = (L + TC - 1) / TC;
    const float* ck = p.ckpt + (size_t)task * (size_t)(nck - 1) * NS * TR;

    const bool fast = vec_u && vec_d && vec_g && vec_B && vec_C;
    constexpr bool tma = TMA;   // host guarantees `fast` whenever it picks the TMA instantiation
    const Stager su = make_row_stager(sm.raw[0][0], (const float*)u_base, p.u_row_stride, t.nrows, lane);
    const Stager sd = make_row_stager(sm.raw[0][1], (const float*)d_base, p.delta_row_stride, t.nrows, lane);
    const Stager sg = make_row_stager(sm.raw[0][2], (const float*)g_base, q.dout_row_stride, t.nrows, lane);
    const Stager sB = make_bc_stager(sm.bc[0][0], (const float*)B_base, p.B_state_stride, N, lane);
    const Stager sC = make_bc_stager(sm.bc[0][1], (const float*)C_base, p.C_state_stride, N, lane);
    Stager16 hu, hd, hg, hB, hC;
    if constexpr (!ASYNC) {
        hu = make_stager16<T>(sm.raw[0][0], 0, u_base, p.u_row_stride, t.nrows, lane);
        hd = make_stager16<T>(sm.raw[0][1], 0, d_base, p.delta_row_stride, t.nrows, lane);
        hg = make_stager16<T>(sm.raw[0][2], 0, g_base, q.dout_row_stride, t.nrows, lane);
        hB = make_stager16<T>(sm.raw[0][0], TR * TC, B_base, p.B_state_stride, N, lane);
        hC = make_stager16<T>(sm.raw[0][1], TR * TC, C_base, p.C_state_stride, N, lane);
    }
    const int lc = (lane & 1) * 4;
    const bool rev = t.rev;
    const int st0 = rev ? TC - 1 - c0 : c0, st1 = rev ? TC - 2 - c0 : c0 + 1;  // scan steps of this lane's two columns
    auto l_lo_of = [&](int c) { return rev ? L - (c + 1) * TC : c * TC; };
    auto prefetch = [&](int c) {  // chunk c (scan order); chunks are visited last -> first
        if (c >= 0) {
            const int buf = c & 1, l_lo = l_lo_of(c);
            if constexpr (!ASYNC) {
                if (fast) {
                    const int l = l_lo + lc;
                    const unsigned off = buf * (unsigned)sizeof(sm.raw[0]);
                    stage8(hu, off, l, L);
                    stage8(hd, off, l, L);
                    stage8(hg, off, l, L);
                    stage8(hB, off, l, L);
                    stage8(hC, off, l, L);
                }
            }
            if (ASYNC) {
                if (fast) {
                    const int l = l_lo + lc;
                    if (tma) {
                        if (lane == 0) {
                            mbar_expect_tx(&sm.bar[buf], 3 * ROW_TILE_BYTES);
                            tma_load_4d(sm.raw[buf][0], &tm.u, l_lo, t.r0, t.g / p.u_group_div, t.b, &sm.bar[buf]);
                            tma_load_4d(sm.raw[buf][1], &tm.delta, l_lo, t.r0, t.g, t.b, &sm.bar[buf]);
                            tma_load_4d(sm.raw[buf][2], &tm.dout, l_lo, t.r0, t.g / (int)q.dout_group_div, t.b, &sm.bar[buf]);
                        }
                    } else {
                        stage16(su, buf * (unsigned)sizeof(sm.raw[0]), l, L, false);
                        stage16(sd, buf * (unsigned)sizeof(sm.raw[0]), l, L, false);
                        stage16(sg, buf * (unsigned)sizeof(sm.raw[0]), l, L, false);
                    }
                    stage16(sB, buf * (unsigned)sizeof(sm.bc[0]), l, L, true);
                    stage16(sC, buf * (unsigned)sizeof(sm.bc[0]), l, L, true);
                } else {
                    stage_rows_slow(sm.raw[buf][0], (const float*)u_base, p.u_row_stride, t.nrows, l_lo, L, lane);
                    stage_rows_slow(sm.raw[buf][1], (const float*)d_base, p.delta_row_stride, t.nrows, l_lo, L, lane);
                    stage_rows_slow(sm.raw[buf][2], (const float*)g_base, q.dout_row_stride, t.nrows, l_lo, L, lane);
                    stage_bc_slow(sm.bc[buf][0], (const float*)B_base, p.B_state_stride, N, l_lo, L, lane);
                    stage_bc_slow(sm.bc[buf][1], (const float*)C_base, p.C_state_stride, N, l_lo, L, lane);
                }
            }
            if (c > 0) stage_ckpt(sm.ck[buf], ck + (size_t)(c - 1) * NS * TR, lane);
        }
        cp_async_commit();
    };
    if (tma) {
        if (lane == 0) {
            mbar_init(&sm.bar[0], 1);
            mbar_init(&sm.bar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }
    // software pipeline with ONE prefetch call site (code size): iterations nck+1 and nck only prefetch
    for (int c = nck + 1; c >= 0; --c) {
        if (c >= nck) {
            prefetch(c - 2);
            continue;
        }
        const int buf = c & 1;
        const int l_lo = l_lo_of(c);
        const int la = l_lo + c0;
        const bool v0 = la >= 0 && la < L, v1 = la + 1 >= 0 && la + 1 < L;
        cp_async_wait<1>();
        if (ASYNC && tma) mbar_wait(&sm.bar[buf], ((nck - 1 - c) >> 1) & 1);   // the ((nck-1-c) >> 1)-th use of this stage
        __syncwarp();
        float uA[2], uB[2], dlA[2], dlB[2], gA[2], gB[2];
        if (ASYNC) {
            const float2 ua = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i, c0)]);
            const float2 ub = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i + 8, c0)]);
            const float2 da = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i, c0)]);
            const float2 db = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i + 8, c0)]);
            const float2 ga = *reinterpret_cast<const float2*>(&sm.raw[buf][2][raw_pos(i, c0)]);
            const float2 gb = *reinterpret_cast<const float2*>(&sm.raw[buf][2][raw_pos(i + 8, c0)]);
            uA[0] = ua.x; uA[1] = ua.y; uB[0] = ub.x; uB[1] = ub.y;
            dlA[0] = da.x; dlA[1] = da.y; dlB[0] = db.x; dlB[1] = db.y;
            gA[0] = ga.x; gA[1] = ga.y; gB[0] = gb.x; gB[1] = gb.y;
        } else if (fast) {
            read_rows16<T>(sm.raw[buf][0], i, sq, uA, uB);
            read_rows16<T>(sm.raw[buf][1], i, sq, dlA, dlB);
            read_rows16<T>(sm.raw[buf][2], i, sq, gA, gB);
            convert_bc16<T>(sm.bc[buf][0], sm.raw[buf][0], lane);
            convert_bc16<T>(sm.bc[buf][1], sm.raw[buf][1], lane);
            __syncwarp();   // the raw slots are reused below for this lane's parked values
        } else {
            fill_bc_sync<T>(sm.bc[buf][0], B_base, p.B_state_stride, N, l_lo, L, lane);
            fill_bc_sync<T>(sm.bc[buf][1], C_base, p.C_state_stride, N, l_lo, L, lane);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const bool v = e ? v1 : v0;
                uA[e] = (okA && v) ? ldg_stream(u_base + (size_t)i * p.u_row_stride + la + e) : 0.f;
                uB[e] = (okB && v) ? ldg_stream(u_base + (size_t)(i + 8) * p.u_row_stride + la + e) : 0.f;
                dlA[e] = (okA && v) ? ldg_stream(d_base + (size_t)i * p.delta_row_stride + la + e) : 0.f;
                dlB[e] = (okB && v) ? ldg_stream(d_base + (size_t)(i + 8) * p.delta_row_stride + la + e) : 0.f;
                gA[e] = (okA && v) ? ldg_stream(g_base + (size_t)i * q.dout_row_stride + la + e) : 0.f;
                gB[e] = (okB && v) ? ldg_stream(g_base + (size_t)(i + 8) * q.dout_row_stride + la + e) : 0.f;
            }
        }
        // ---- prologue (once per element): delta', its sigmoid, the gated upstream gradient ----
        float sgA[2], sgB[2], dzA[2], dzB[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool v = e ? v1 : v0;
            float a = dlA[e] + biasA, b = dlB[e] + biasB, sa = 1.f, sb = 1.f;
            if (softplus) {
                const SoftplusSig ra = softplus_sigmoid(a), rb = softplus_sigmoid(b);
                a = ra.sp; sa = ra.sig; b = rb.sp; sb = rb.sig;
            }
            const bool va = okA && v, vb = okB && v;
            dlA[e] = va ? a : 0.f; sgA[e] = va ? sa : 0.f;  // identity steps (u and dout are already zero there)
            dlB[e] = vb ? b : 0.f; sgB[e] = vb ? sb : 0.f;
            if (HAS_Z) {
                const float za = va ? ldg_stream(z_base + (size_t)i * p.z_row_stride + la + e) : 0.f;
                const float zb = vb ? ldg_stream(z_base + (size_t)(i + 8) * p.z_row_stride + la + e) : 0.f;
                const float s_a = sigmoidf_(za), s_b = sigmoidf_(zb);
                dzA[e] = gA[e] * s_a * (1.f + za * (1.f - s_a));  // dout * d silu(z)/dz
                dzB[e] = gB[e] * s_b * (1.f + zb * (1.f - s_b));
                gA[e] *= za * s_a;                                 // dout * silu(z)
                gB[e] *= zb * s_b;
            }
            const int st = e ? st1 : st0;   // the exchange tile is indexed by scan step
            *reinterpret_cast<float2*>(&sm.ex[0][st * EXS + 2 * i]) = make_float2(dlA[e], dlB[e]);
            *reinterpret_cast<float2*>(&sm.ex[1][st * EXS + 2 * i]) = make_float2(dlA[e] * uA[e], dlB[e] * uB[e]);
            *reinterpret_cast<float2*>(&sm.ex[2][st * EXS + 2 * i]) = make_float2(gA[e], gB[e]);
        }
        // park what the epilogue needs where only this lane looks (its own slots of the raw tiles)
        if (!ASYNC) {
            *reinterpret_cast<float2*>(&sm.raw[buf][0][raw_pos(i, c0)]) = make_float2(uA[0], uA[1]);
            *reinterpret_cast<float2*>(&sm.raw[buf][0][raw_pos(i + 8, c0)]) = make_float2(uB[0], uB[1]);
        }
        *reinterpret_cast<float2*>(&sm.raw[buf][1][raw_pos(i, c0)]) = make_float2(sgA[0], sgA[1]);
        *reinterpret_cast<float2*>(&sm.raw[buf][1][raw_pos(i + 8, c0)]) = make_float2(sgB[0], sgB[1]);
        if (HAS_Z) {
            *reinterpret_cast<float2*>(&sm.raw[buf][2][raw_pos(i, c0)]) = make_float2(dzA[0], dzA[1]);
            *reinterpret_cast<float2*>(&sm.raw[buf][2][raw_pos(i + 8, c0)]) = make_float2(dzB[0], dzB[1]);
        }
        __syncwarp();
        float2 dl2[TC], q2[TC], go2[TC], s1[TC], s2[TC], yacc[HAS_Z ? TC : 1];
#pragma unroll
        for (int cc = 0; cc < TC; ++cc) {
            dl2[cc] = *reinterpret_cast<const float2*>(&sm.ex[0][cc * EXS + 2 * i]);
            q2[cc] = *reinterpret_cast<const float2*>(&sm.ex[1][cc * EXS + 2 * i]);
            go2[cc] = *reinterpret_cast<const float2*>(&sm.ex[2][cc * EXS + 2 * i]);
            s1[cc] = make_float2(0.f, 0.f);
            s2[cc] = make_float2(0.f, 0.f);
            if constexpr (HAS_Z) yacc[cc] = make_float2(0.f, 0.f);
        }

        // ---- this lane's 4 states, one after the other.  The scan direction is a RUNTIME property (tiles indexed by
        //      scan step): with one compile-time body per direction the two unrolled copies evicted each other from the
        //      32 KB instruction cache whenever an SM ran both kinds of task (measured: +25 % time under SS2D's rev_mask) ----
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
            const int n = sq * SPT + j;
            const float2 A2j = sm.A2[j][lane];
            float2 xm1 = make_float2(0.f, 0.f);
            if (c > 0) xm1 = *reinterpret_cast<const float2*>(&sm.ck[buf][sq * CKS + j * 16 + 2 * i]);
            float Bv[TC];
            load8_steps(&sm.bc[buf][0][sq * BCS + j * TC], rev, Bv);
            // forward recompute of the chunk from its checkpoint
            float2 a[TC], x[TC];
            {
                float2 xs = xm1;
#pragma unroll
                for (int s = 0; s < TC; ++s) {
                    const int cc = s;
                    a[s] = ex2_2(__fmul2_rn(dl2[cc], A2j));
                    const float2 qB = make_float2(q2[cc].x * Bv[cc], q2[cc].y * Bv[cc]);
                    xs = __ffma2_rn(a[s], xs, qB);
                    x[s] = xs;
                }
            }
            // adjoint recurrence, last step first.  gn = a_{s+1} * (adjoint of x_{s+1})
            float Cv[TC];
            load8_steps(&sm.bc[buf][1][sq * BCS + j * TC], rev, Cv);
            float2 gn = sm.h[j][lane];
            float2 dAp = make_float2(0.f, 0.f);
            float vB[TC], vC[TC];
#pragma unroll
            for (int s = TC - 1; s >= 0; --s) {
                const int cc = s;
                const float2 xprev = s > 0 ? x[s - 1] : xm1;
                float2 g;
                g.x = fmaf(go2[cc].x, Cv[cc], gn.x);
                g.y = fmaf(go2[cc].y, Cv[cc], gn.y);
                vC[cc] = fmaf(go2[cc].y, x[s].y, go2[cc].x * x[s].x);  // sum over the row pair
                vB[cc] = fmaf(g.y, q2[cc].y, g.x * q2[cc].x);
                s1[cc].x = fmaf(g.x, Bv[cc], s1[cc].x);
                s1[cc].y = fmaf(g.y, Bv[cc], s1[cc].y);
                gn = __fmul2_rn(a[s], g);
                const float2 wv = __fmul2_rn(gn, xprev);
                s2[cc] = __ffma2_rn(A2j, wv, s2[cc]);  // A * log2(e): rescaled by ln 2 in the epilogue
                dAp = __ffma2_rn(wv, dl2[cc], dAp);
                if constexpr (HAS_Z) {
                    yacc[cc].x = fmaf(Cv[cc], x[s].x, yacc[cc].x);
                    yacc[cc].y = fmaf(Cv[cc], x[s].y, yacc[cc].y);
                }
            }
            sm.h[j][lane] = gn;
            sm.dA[j][lane] = __fadd2_rn(sm.dA[j][lane], dAp);
            // dB / dC: sum over the 16 rows, lane i ends with column i: one RED per (state, quantity)
            const float rB = rs8_rows(vB, lane);   // (a shared-memory transposition was measured slower: LSU wavefronts)
            const float rC = rs8_rows(vC, lane);
            const int lcol = l_lo + (rev ? TC - 1 - i : i);   // lane i holds scan step i
            if (n < N && (unsigned)lcol < (unsigned)L) {
                atomicAdd(dB_base + n * dBs + lcol, rB);
                atomicAdd(dC_base + n * dCs + lcol, rC);
            }
        }

        // ---- per-element gradients: sums over the 16 states, then this lane's 2 rows x 2 columns ----
        float2 t1a, t1b, t2a, t2b, tya = make_float2(0.f, 0.f), tyb = tya;
        reduce_states(sm.rd, s1, lane, st0, st1, t1a, t1b);
        __syncwarp();
        reduce_states(sm.rd, s2, lane, st0, st1, t2a, t2b);
        if constexpr (HAS_Z) {
            __syncwarp();
            reduce_states(sm.rd, yacc, lane, st0, st1, tya, tyb);
        }
        {
            const float2 ua = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i, c0)]);
            const float2 ub = *reinterpret_cast<const float2*>(&sm.raw[buf][0][raw_pos(i + 8, c0)]);
            const float2 sa = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i, c0)]);
            const float2 sb = *reinterpret_cast<const float2*>(&sm.raw[buf][1][raw_pos(i + 8, c0)]);
            const float2 dl0 = *reinterpret_cast<const float2*>(&sm.ex[0][st0 * EXS + 2 * i]);        // (row A, row B) of column c0
            const float2 dl1 = *reinterpret_cast<const float2*>(&sm.ex[0][st1 * EXS + 2 * i]);
            const float2 go0 = *reinterpret_cast<const float2*>(&sm.ex[2][st0 * EXS + 2 * i]);
            const float2 go1 = *reinterpret_cast<const float2*>(&sm.ex[2][st1 * EXS + 2 * i]);
            const float duA0 = fmaf(dl0.x, t1a.x, DA * go0.x), duA1 = fmaf(dl1.x, t1b.x, DA * go1.x);
            const float duB0 = fmaf(dl0.y, t1a.y, DB * go0.y), duB1 = fmaf(dl1.y, t1b.y, DB * go1.y);
            // chain rule through softplus: sg = sigmoid(delta + bias) (1 without softplus, 0 off-range)
            const float ddA0 = fmaf(ua.x, t1a.x, t2a.x * kLn2) * sa.x, ddA1 = fmaf(ua.y, t1b.x, t2b.x * kLn2) * sa.y;
            const float ddB0 = fmaf(ub.x, t1a.y, t2a.y * kLn2) * sb.x, ddB1 = fmaf(ub.y, t1b.y, t2b.y * kLn2) * sb.y;
            dbias_A += ddA0 + ddA1;
            dbias_B += ddB0 + ddB1;
            dD_A = fmaf(go0.x, ua.x, fmaf(go1.x, ua.y, dD_A));
            dD_B = fmaf(go0.y, ub.x, fmaf(go1.y, ub.y, dD_B));
            store_pair<T>(du_base + (size_t)i * q.du_row_stride + la, duA0, duA1, okA && v0, okA && v1, vec_du);
            store_pair<T>(du_base + (size_t)(i + 8) * q.du_row_stride + la, duB0, duB1, okB && v0, okB && v1, vec_du);
            store_pair<T>(dd_base + (size_t)i * q.ddelta_row_stride + la, ddA0, ddA1, okA && v0, okA && v1, vec_dd);
            store_pair<T>(dd_base + (size_t)(i + 8) * q.ddelta_row_stride + la, ddB0, ddB1, okB && v0, okB && v1, vec_dd);
            if (HAS_Z) {
                const float2 za = *reinterpret_cast<const float2*>(&sm.raw[buf][2][raw_pos(i, c0)]);
                const float2 zb = *reinterpret_cast<const float2*>(&sm.raw[buf][2][raw_pos(i + 8, c0)]);
                store_pair<T>(dz_base + (size_t)i * q.dz_row_stride + la, za.x * fmaf(DA, ua.x, tya.x), za.y * fmaf(DA, ua.y, tyb.x),
                              okA && v0, okA && v1, vec_dz);
                store_pair<T>(dz_base + (size_t)(i + 8) * q.dz_row_stride + la, zb.x * fmaf(DB, ub.x, tya.y),
                              zb.y * fmaf(DB, ub.y, tyb.y), okB && v0, okB && v1, vec_dz);
            }
        }
        if (tma) fence_proxy_async();
        __syncwarp();  // every lane is done with this chunk's tiles
        prefetch(c - 2);
    }
    cp_async_wait<0>();

#pragma unroll
    for (int j = 0; j < SPT; ++j) {
        const int n = sq * SPT + j;
        if (n < N) {
            const float2 v = sm.dA[j][lane];
            if (okA) atomicAdd(q.dA + (size_t)dA_ * N + n, v.x);
            if (okB) atomicAdd(q.dA + (size_t)dB_ * N + n, v.y);
        }
    }
    // per-row sums: the four state-quad lanes of a row pair each hold two columns' worth
#pragma unroll
    for (int m = 8; m <= 16; m <<= 1) {
        dD_A += __shfl_xor_sync(0xffffffffu, dD_A, m);
        dD_B += __shfl_xor_sync(0xffffffffu, dD_B, m);
        dbias_A += __shfl_xor_sync(0xffffffffu, dbias_A, m);
        dbias_B += __shfl_xor_sync(0xffffffffu, dbias_B, m);
    }
    if (sq == 0) {
        if (okA) {
            if (q.ddelta_bias) atomicAdd(q.ddelta_bias + dA_, dbias_A);
            if (q.dD) atomicAdd(q.dD + dA_, dD_A);
        }
        if (okB) {
            if (q.ddelta_bias) atomicAdd(q.ddelta_bias + dB_, dbias_B);
            if (q.dD) atomicAdd(q.dD + dB_, dD_B);
        }
    }
}

template <typename T, bool HAS_Z, bool TMA>
__global__ void __launch_bounds__(WPB * 32, 12) sscan_bwd_kernel(const __grid_constant__ b200_sscan_bwd_params q, const __grid_constant__ RowMaps tm) {
    __shared__ __align__(1024) BwdWarpSmem sm;
    const int lane = threadIdx.x;
    const long long task = blockIdx.x;
    const Task t = decode_task(q.f, task);
    sscan_bwd_body<T, HAS_Z, TMA>(q, tm, t, task, sm, lane);
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
static int validate(const b200_sscan_fwd_params* p) {
    B200_REQUIRE(p != nullptr, "b200_sscan: params is NULL");
    B200_REQUIRE(p->batch > 0 && p->dim > 0 && p->seqlen > 0, "b200_sscan: batch/dim/seqlen must be positive (got %d/%d/%d)",
                 p->batch, p->dim, p->seqlen);
    B200_REQUIRE(p->dstate >= 1 && p->dstate <= B200_SSCAN_MAX_DSTATE, "b200_sscan: dstate %d outside [1, %d]", p->dstate,
                 B200_SSCAN_MAX_DSTATE);
    B200_REQUIRE(p->dstate <= NS, "b200_sscan: dstate %d > %d is not implemented in this build", p->dstate, NS);
    B200_REQUIRE(p->n_groups >= 1 && p->dim % p->n_groups == 0, "b200_sscan: dim %d is not divisible by n_groups %d", p->dim,
                 p->n_groups);
    B200_REQUIRE(p->io_dtype >= B200_F32 && p->io_dtype <= B200_F16, "b200_sscan: bad io_dtype %d", p->io_dtype);
    B200_REQUIRE(p->rev_mask == 0 || p->n_groups <= 32, "b200_sscan: rev_mask needs n_groups <= 32");
    B200_REQUIRE(p->u_group_div >= 1 && p->n_groups % p->u_group_div == 0, "b200_sscan: u_group_div %d must be >= 1 and divide n_groups %d",
                 p->u_group_div, p->n_groups);
    B200_REQUIRE((long long)p->dstate * p->seqlen < (1ll << 31), "b200_sscan: dstate * seqlen must be < 2^31");
    B200_REQUIRE(p->u && p->delta && p->A && p->B && p->C, "b200_sscan: u/delta/A/B/C must be non-NULL");
    B200_REQUIRE(p->ckpt == nullptr || p->ckpt_every == TC, "b200_sscan: ckpt_every must be %d", TC);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(p->ckpt) & 15) == 0, "b200_sscan: ckpt must be 16-byte aligned");
    return 0;
}

static long long n_tasks(const b200_sscan_fwd_params* p) {
    const int rpg = p->dim / p->n_groups;
    return (long long)p->batch * p->n_groups * tiles_per_group(rpg);
}

// static shared memory only, but 12-16 resident warp-CTAs need the large carve-out
template <typename K> static void prefer_smem(K kernel) {
    (void)func_attr_per_device((const void*)kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

// ---- tensor maps for the TMA row path ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
    static const EncodeTiledFn fn = [] {
        const char* on = getenv("B200_SSCAN_TMA");   // opt-in: measured 5 % slower than the LDGSTS staging at 512-byte boxes
        if (!on || on[0] != '1') return (EncodeTiledFn) nullptr;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qr) != cudaSuccess ||
            qr != cudaDriverEntryPointSuccess)
            ptr = nullptr;
        (void)cudaGetLastError();
        return (EncodeTiledFn)ptr;
    }();
    return fn;
}
// fp32 activation tensor viewed as (L, rows per group, groups, batch); box = (8 steps, 16 rows, 1, 1), SWIZZLE_32B
static bool make_row_map(CUtensorMap* m, const void* base, int L, int rpg, int groups, int batch, int64_t row_stride,
                         int64_t group_stride, int64_t batch_stride) {
    const EncodeTiledFn enc = encode_tiled();
    if (!enc || (L & 3) || (reinterpret_cast<uintptr_t>(base) & 15) || (row_stride & 3) || (group_stride & 3) || (batch_stride & 3))
        return false;
    if (row_stride <= 0 || group_stride <= 0 || batch_stride <= 0) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)L, (cuuint64_t)rpg, (cuuint64_t)groups, (cuuint64_t)batch};
    const cuuint64_t strides[3] = {(cuuint64_t)row_stride * 4, (cuuint64_t)group_stride * 4, (cuuint64_t)batch_stride * 4};
    for (int k = 0; k < 3; ++k)
        if (strides[k] >= (1ull << 40)) return false;
    const cuuint32_t box[4] = {TC, TR, 1, 1}, estr[4] = {1, 1, 1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static bool bc_vec_ok(const void* ptr, int64_t state_stride, int64_t batch_stride, int64_t group_stride) {
    return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (state_stride & 3) == 0 && (batch_stride & 3) == 0 && (group_stride & 3) == 0;
}
static bool make_fwd_maps(RowMaps* tm, const b200_sscan_fwd_params* p) {
    if (p->io_dtype != B200_F32 || encode_tiled() == nullptr) return false;
    const int rpg = p->dim / p->n_groups;
    if (p->n_groups % p->u_group_div) return false;
    // the kernel's TMA instantiation assumes its 16-byte B/C staging is legal too
    if (!bc_vec_ok(p->B, p->B_state_stride, p->B_batch_stride, p->B_group_stride) ||
        !bc_vec_ok(p->C, p->C_state_stride, p->C_batch_stride, p->C_group_stride))
        return false;
    return make_row_map(&tm->u, p->u, p->seqlen, rpg, p->n_groups / p->u_group_div, p->batch, p->u_row_stride, p->u_group_stride,
                        p->u_batch_stride) &&
           make_row_map(&tm->delta, p->delta, p->seqlen, rpg, p->n_groups, p->batch, p->delta_row_stride,
                        p->delta_group_stride, p->delta_batch_stride);
}

// b200_sscan_last_variant(): 1 = sscan.cu, 2 = sscan2.cu, 3 = sscan.cu with the TMA row staging (include/b200_ssm.h)
static thread_local int g_last_variant = 0;

template <typename T>
static int launch_fwd(const b200_sscan_fwd_params* p, cudaStream_t st) {
    const long long nt = n_tasks(p);
    const unsigned grid = (unsigned)((nt + WPB - 1) / WPB);
    RowMaps tm;
    memset(&tm, 0, sizeof(tm));
    const bool use_tma = sizeof(T) == 4 && make_fwd_maps(&tm, p);
    g_last_variant = use_tma ? 3 : 1;
    if (use_tma) {
        if (p->z) sscan_fwd_kernel<T, true, sizeof(T) == 4><<<grid, WPB * 32, 0, st>>>(*p, tm);
        else sscan_fwd_kernel<T, false, sizeof(T) == 4><<<grid, WPB * 32, 0, st>>>(*p, tm);
    } else {
        if (p->z) sscan_fwd_kernel<T, true, false><<<grid, WPB * 32, 0, st>>>(*p, tm);
        else sscan_fwd_kernel<T, false, false><<<grid, WPB * 32, 0, st>>>(*p, tm);
    }
    return check_launch("sscan_fwd_kernel");
}

template <typename T>
static int launch_bwd(const b200_sscan_bwd_params* q, cudaStream_t st) {
    prefer_smem(sscan_bwd_kernel<T, true, false>);    // remembered per (kernel, device)
    prefer_smem(sscan_bwd_kernel<T, false, false>);
    prefer_smem(sscan_bwd_kernel<T, true, sizeof(T) == 4>);
    prefer_smem(sscan_bwd_kernel<T, false, sizeof(T) == 4>);
    const long long nt = n_tasks(&q->f);
    const unsigned grid = (unsigned)((nt + WPB - 1) / WPB);
    RowMaps tm;
    memset(&tm, 0, sizeof(tm));
    const int rpg = q->f.dim / q->f.n_groups;
    const int use_tma = (make_fwd_maps(&tm, &q->f) && q->f.n_groups % (int)q->dout_group_div == 0 &&
                         make_row_map(&tm.dout, q->dout, q->f.seqlen, rpg, q->f.n_groups / (int)q->dout_group_div, q->f.batch,
                                      q->dout_row_stride, q->dout_group_stride, q->dout_batch_stride))
                            ? 1
                            : 0;
    g_last_variant = use_tma && sizeof(T) == 4 ? 3 : 1;
    if (use_tma && sizeof(T) == 4) {
        if (q->f.z) sscan_bwd_kernel<T, true, sizeof(T) == 4><<<grid, WPB * 32, 0, st>>>(*q, tm);
        else sscan_bwd_kernel<T, false, sizeof(T) == 4><<<grid, WPB * 32, 0, st>>>(*q, tm);
    } else {
        if (q->f.z) sscan_bwd_kernel<T, true, false><<<grid, WPB * 32, 0, st>>>(*q, tm);
        else sscan_bwd_kernel<T, false, false><<<grid, WPB * 32, 0, st>>>(*q, tm);
    }
    return check_launch("sscan_bwd_kernel");
}

}  // namespace b200

namespace b200 {
namespace v2 {   // sscan2.cu: TMA-staged kernels for fp32 tensors with 16-byte aligned layouts
bool try_fwd(const b200_sscan_fwd_params* p, cudaStream_t st, int* rc);
bool try_bwd(const b200_sscan_bwd_params* q, cudaStream_t st, int* rc);
}
}

using namespace b200;

extern "C" int b200_sscan_last_variant(void) { return g_last_variant; }

extern "C" size_t b200_sscan_ckpt_bytes(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate, int32_t n_groups,
                                        int32_t ckpt_every) {
    (void)dstate;
    if (batch <= 0 || dim <= 0 || seqlen <= 0 || n_groups <= 0 || dim % n_groups || ckpt_every <= 0) return 0;
    const int rpg = dim / n_groups;
    const size_t tasks = (size_t)batch * n_groups * tiles_per_group(rpg);
    const size_t nck = (seqlen + ckpt_every - 1) / ckpt_every;
    const size_t bytes = tasks * (nck - 1) * NS * TR * sizeof(float);
    return bytes ? bytes : 16;
}

extern "C" int b200_sscan_fwd(const b200_sscan_fwd_params* p, b200_stream_t stream) {
    if (int rc = validate(p)) return rc;
    B200_REQUIRE(p->out != nullptr, "b200_sscan_fwd: out is NULL");
    B200_REQUIRE(n_tasks(p) < (1ll << 31), "b200_sscan_fwd: too many rows");
    cudaStream_t st = (cudaStream_t)stream;
    {
        int rc = 0;
        if (v2::try_fwd(p, st, &rc)) {
            g_last_variant = 2;
            return rc;
        }
    }
    switch (p->io_dtype) {
        case B200_F32: return launch_fwd<float>(p, st);
        case B200_BF16: return launch_fwd<__nv_bfloat16>(p, st);
        default: return launch_fwd<__half>(p, st);
    }
}

extern "C" int b200_sscan_bwd(const b200_sscan_bwd_params* q, b200_stream_t stream) {
    B200_REQUIRE(q != nullptr, "b200_sscan_bwd: params is NULL");
    if (int rc = validate(&q->f)) return rc;
    B200_REQUIRE(q->f.ckpt != nullptr, "b200_sscan_bwd: the forward checkpoints (f.ckpt) are required");
    B200_REQUIRE(q->dout && q->du && q->ddelta && q->dA && q->dB && q->dC, "b200_sscan_bwd: dout/du/ddelta/dA/dB/dC must be non-NULL");
    B200_REQUIRE((q->f.z == nullptr) == (q->dz == nullptr), "b200_sscan_bwd: dz must be given exactly when z is");
    B200_REQUIRE(q->dout_group_div >= 1 && q->f.n_groups % (int)q->dout_group_div == 0,
                 "b200_sscan_bwd: dout_group_div must be >= 1 and divide n_groups");
    B200_REQUIRE(q->dB_state_stride >= q->f.seqlen && q->dC_state_stride >= q->f.seqlen &&
                     (long long)q->f.dstate * q->dB_state_stride < (1ll << 31) && (long long)q->f.dstate * q->dC_state_stride < (1ll << 31),
                 "b200_sscan_bwd: dB/dC state strides must be in [seqlen, 2^31 / dstate)");
    B200_REQUIRE(n_tasks(&q->f) < (1ll << 31), "b200_sscan_bwd: too many rows");
    cudaStream_t st = (cudaStream_t)stream;
    {
        int rc = 0;
        if (v2::try_bwd(q, st, &rc)) {
            g_last_variant = 2;
            return rc;
        }
    }
    switch (q->f.io_dtype) {
        case B200_F32: return launch_bwd<float>(q, st);
        case B200_BF16: return launch_bwd<__nv_bfloat16>(q, st);
        default: return launch_bwd<__half>(q, st);
    }
}
