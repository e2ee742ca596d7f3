// conv1d.cu -- causal depth-wise conv1d (+ bias, + SiLU) forward and backward, sm_100a.
//
// The conv of the Mamba-2 mixer (causal-conv1d's causal_conv1d_fn, as mamba_ssm 2.2.2's mamba_split_conv1d_scan_combined runs it
// over the xBC slice of in_proj's output).  Channel c of a (batch, L, C) channel-last input, width W in 2..4, all arithmetic fp32:
//
//   a[t] = bias[c] + sum_k w[c, k] * x[t - (W-1) + k] * m(t - (W-1) + k, t),     y[t] = silu(a[t]) or a[t]
//
// x before the sequence start is zero, and m(s, t) = 1 unless seq_idx is given and seq_idx[s] != seq_idx[t] (a packed row: no tap
// crosses a sequence boundary).  Backward, from the fp32 gradient dy of y, g[t] = dy[t] * act'(a[t]) with a[t] recomputed:
//
//   dx[s] = sum_k w[k] g[s + (W-1) - k] m(s, s + (W-1) - k)     dw[k] = sum_t g[t] x[t - (W-1) + k] m(.)     db = sum_t g[t]
//
// Layout: CTA (channel tile, time tile of CV_TL steps, batch row); each of its CV_THREADS threads owns V consecutive channels and
// walks the tile's time steps in order, keeping the last W-1 inputs (and seq ids) in registers, so every input is read once plus a
// W-1 halo per tile.  Loads of CV_U steps are issued before their arithmetic.  The backward walks the tile plus W-1 steps of the next
// one (their g completes the tile's last dx) and carries the W partial dx sums of the positions still open; d(weight) / d(bias) of
// the tile's steps stay in registers and each thread writes them as its share of one partial row per CTA (no atomics: the same
// grid gives the same sums, bitwise).  x, y, dx are read and written in place with their own batch and time strides (the xBC slice
// of in_proj's output, whose row pitch is often not a multiple of 4 elements); V is the widest vector every base and stride allows.
#include "common.cuh"

namespace b200 {

constexpr int CV_THREADS = 128;
constexpr int CV_TL = 64;       // time steps per CTA
constexpr int CV_U = 4;         // steps whose loads are issued together

struct ConvArgs {
    const void* x;
    const float* w;
    const float* b;
    const int32_t* seq;
    void* y;          // forward output
    const float* dy;  // backward input (fp32)
    void* dx;
    float* dwp;
    float* dbp;
    int64_t xb, xl, sb, sl, yb, yl, gb, gl, dxb, dxl;
    int L, C, x_dt, y_dt, silu;
};

__device__ __forceinline__ float cv_act(float a, int silu) { return silu ? a / (1.f + expf(-a)) : a; }

template <int V>
__device__ __forceinline__ void cv_ld_f32(const float* p, float* v) {
    if constexpr (V == 4) {
        const float4 u = __ldcs(reinterpret_cast<const float4*>(p));
        v[0] = u.x, v[1] = u.y, v[2] = u.z, v[3] = u.w;
    } else if constexpr (V == 2) {
        const float2 u = __ldcs(reinterpret_cast<const float2*>(p));
        v[0] = u.x, v[1] = u.y;
    } else {
        v[0] = __ldcs(p);
    }
}

template <int W, int V, bool SEQ>
__global__ void __launch_bounds__(CV_THREADS) causal_conv1d_fwd_kernel(const ConvArgs a) {
    const int c = (blockIdx.x * CV_THREADS + threadIdx.x) * V;
    if (c >= a.C) return;
    const int64_t b = blockIdx.z;
    const int t0 = blockIdx.y * CV_TL, t1 = min(t0 + CV_TL, a.L);
    float w[V][W], bias[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
#pragma unroll
        for (int k = 0; k < W; ++k) w[j][k] = __ldg(a.w + (int64_t)(c + j) * W + k);
        bias[j] = a.b ? __ldg(a.b + c + j) : 0.f;
    }
    const int64_t xo = b * a.xb + c, yo = b * a.yb + c, so = b * a.sb;
    float h[W][V];     // h[k]: x at t - (W-1) + k
    int sid[W];
#pragma unroll
    for (int k = 0; k < W - 1; ++k) {
        const int t = t0 - (W - 1) + k;
        uint32_t r[V];
        if (t >= 0) {
            rn_ld<V>(a.x, xo + t * a.xl, a.x_dt, r);
            rn_cvt<V>(r, a.x_dt, h[k]);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) h[k][j] = 0.f;
        }
        sid[k] = SEQ && t >= 0 ? __ldg(a.seq + so + t * a.sl) : -1;
    }
    for (int tb = t0; tb < t1; tb += CV_U) {
        uint32_t r[CV_U][V];
        int sq[CV_U];
#pragma unroll
        for (int u = 0; u < CV_U; ++u) {
            const int t = tb + u;
            if (t < t1) {
                rn_ld<V>(a.x, xo + t * a.xl, a.x_dt, r[u]);
                if (SEQ) sq[u] = __ldg(a.seq + so + t * a.sl);
            }
        }
#pragma unroll
        for (int u = 0; u < CV_U; ++u) {
            const int t = tb + u;
            if (t < t1) {
                rn_cvt<V>(r[u], a.x_dt, h[W - 1]);
                sid[W - 1] = SEQ ? sq[u] : 0;
                float o[V];
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    float acc = bias[j];
#pragma unroll
                    for (int k = 0; k < W; ++k)
                        if (!SEQ || k == W - 1 || sid[k] == sid[W - 1]) acc = fmaf(w[j][k], h[k][j], acc);
                    o[j] = cv_act(acc, a.silu);
                }
                rn_st<V>(a.y, yo + t * a.yl, a.y_dt, o);
#pragma unroll
                for (int k = 0; k < W - 1; ++k) {
                    sid[k] = sid[k + 1];
#pragma unroll
                    for (int j = 0; j < V; ++j) h[k][j] = h[k + 1][j];
                }
            }
        }
    }
}

template <int W, int V, bool SEQ>
__global__ void __launch_bounds__(CV_THREADS) causal_conv1d_bwd_kernel(const ConvArgs a) {
    const int c = (blockIdx.x * CV_THREADS + threadIdx.x) * V;
    if (c >= a.C) return;
    const int64_t b = blockIdx.z;
    const int t0 = blockIdx.y * CV_TL, t1 = min(t0 + CV_TL, a.L);
    const int te = min(t1 + W - 1, a.L);       // the steps whose g reaches dx of [t0, t1)
    float w[V][W], bias[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
#pragma unroll
        for (int k = 0; k < W; ++k) w[j][k] = __ldg(a.w + (int64_t)(c + j) * W + k);
        bias[j] = a.b ? __ldg(a.b + c + j) : 0.f;
    }
    const int64_t xo = b * a.xb + c, go = b * a.gb + c, dxo = b * a.dxb + c, so = b * a.sb;
    float h[W][V], pdx[W][V], dw[V][W], db[V];   // pdx[k]: the open dx sum of position t - (W-1) + k
    int sid[W];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        db[j] = 0.f;
#pragma unroll
        for (int k = 0; k < W; ++k) dw[j][k] = pdx[k][j] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < W - 1; ++k) {
        const int t = t0 - (W - 1) + k;
        uint32_t r[V];
        if (t >= 0) {
            rn_ld<V>(a.x, xo + t * a.xl, a.x_dt, r);
            rn_cvt<V>(r, a.x_dt, h[k]);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) h[k][j] = 0.f;
        }
        sid[k] = SEQ && t >= 0 ? __ldg(a.seq + so + t * a.sl) : -1;
    }
    // te - t0 steps, then the W-1 positions still open at the row's end are closed by steps of g = 0
    const int tz = t1 + W - 1;
    for (int tb = t0; tb < tz; tb += CV_U) {
        uint32_t r[CV_U][V];
        float gv[CV_U][V];
        int sq[CV_U];
#pragma unroll
        for (int u = 0; u < CV_U; ++u) {
            const int t = tb + u;
            if (t < te) {
                rn_ld<V>(a.x, xo + t * a.xl, a.x_dt, r[u]);
                cv_ld_f32<V>(a.dy + go + t * a.gl, gv[u]);
                if (SEQ) sq[u] = __ldg(a.seq + so + t * a.sl);
            }
        }
#pragma unroll
        for (int u = 0; u < CV_U; ++u) {
            const int t = tb + u;
            if (t < tz) {
                const bool live = t < te;
                if (live) {
                    rn_cvt<V>(r[u], a.x_dt, h[W - 1]);
                    sid[W - 1] = SEQ ? sq[u] : 0;
                } else {
#pragma unroll
                    for (int j = 0; j < V; ++j) h[W - 1][j] = 0.f;
                    sid[W - 1] = sid[W - 2];
                }
                bool m[W];
#pragma unroll
                for (int k = 0; k < W; ++k) m[k] = !SEQ || k == W - 1 || sid[k] == sid[W - 1];
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    float g = 0.f;
                    if (live) {
                        float acc = bias[j];
#pragma unroll
                        for (int k = 0; k < W; ++k)
                            if (m[k]) acc = fmaf(w[j][k], h[k][j], acc);
                        g = gv[u][j];
                        if (a.silu) {
                            const float s = 1.f / (1.f + expf(-acc));
                            g *= s * (1.f + acc * (1.f - s));
                        }
                    }
                    if (t < t1) {
                        db[j] += g;
#pragma unroll
                        for (int k = 0; k < W; ++k)
                            if (m[k]) dw[j][k] = fmaf(g, h[k][j], dw[j][k]);
                    }
#pragma unroll
                    for (int k = 0; k < W; ++k)
                        if (m[k]) pdx[k][j] = fmaf(w[j][k], g, pdx[k][j]);
                }
                const int s0 = t - (W - 1);            // its last contribution is this step's
                if (s0 >= t0) rn_st<V>(a.dx, dxo + s0 * a.dxl, a.x_dt, pdx[0]);
#pragma unroll
                for (int k = 0; k < W - 1; ++k) {
                    sid[k] = sid[k + 1];
#pragma unroll
                    for (int j = 0; j < V; ++j) {
                        h[k][j] = h[k + 1][j];
                        pdx[k][j] = pdx[k + 1][j];
                    }
                }
#pragma unroll
                for (int j = 0; j < V; ++j) pdx[W - 1][j] = 0.f;
            }
        }
    }
    const int64_t row = b * gridDim.y + blockIdx.y;
#pragma unroll
    for (int j = 0; j < V; ++j) {
#pragma unroll
        for (int k = 0; k < W; ++k) a.dwp[(row * a.C + c + j) * W + k] = dw[j][k];
        if (a.dbp) a.dbp[row * a.C + c + j] = db[j];
    }
}

// One decoding step (causal_conv1d_update): a thread per (channel, batch row) walks the seqlen new inputs with the last W-1 values
// of v = cat(conv_state, x) in registers, then shifts conv_state left by seqlen in place.  The shift reads column j + seqlen before
// it writes column j, and every column it reads at or after j + seqlen is still unwritten, so one thread needs no staging.
struct ConvUpdateArgs {
    const void* x;
    void* st;
    const void* w;
    const void* b;
    void* y;
    int64_t xb, xc, xl, sb, sc, sl, wc, wk, bs, yb, yc, yl;
    int C, L, S, dt, w_dt, b_dt, silu;
};

__device__ __forceinline__ float cv_ld1(const void* base, int64_t idx, int dt) {
    uint32_t r[1];
    float v[1];
    rn_ld<1>(base, idx, dt, r);
    rn_cvt<1>(r, dt, v);
    return v[0];
}

template <int W>
__global__ void __launch_bounds__(CV_THREADS) causal_conv1d_update_kernel(const ConvUpdateArgs a) {
    const int c = blockIdx.x * CV_THREADS + threadIdx.x;
    if (c >= a.C) return;
    const int64_t b = blockIdx.y;
    const int64_t xo = b * a.xb + c * a.xc, so = b * a.sb + c * a.sc, yo = b * a.yb + c * a.yc;
    float w[W], h[W];
#pragma unroll
    for (int k = 0; k < W; ++k) w[k] = cv_ld1(a.w, c * a.wc + k * a.wk, a.w_dt);
    const float bias = a.b ? cv_ld1(a.b, c * a.bs, a.b_dt) : 0.f;
#pragma unroll
    for (int k = 0; k < W - 1; ++k) h[k] = cv_ld1(a.st, so + (a.S - (W - 1) + k) * a.sl, a.dt);
    for (int t = 0; t < a.L; ++t) {
        h[W - 1] = cv_ld1(a.x, xo + t * a.xl, a.dt);
        float acc = bias;
#pragma unroll
        for (int k = 0; k < W; ++k) acc = fmaf(w[k], h[k], acc);
        const float o[1] = {cv_act(acc, a.silu)};
        rn_st<1>(a.y, yo + t * a.yl, a.dt, o);
#pragma unroll
        for (int k = 0; k < W - 1; ++k) h[k] = h[k + 1];
    }
    // conv_state <- the last S columns of cat(conv_state, x): column j takes v[j + L] (a 16-bit value survives the fp32 round trip)
#pragma unroll 1   // unrolled, this loop makes ptxas spill
    for (int j = 0; j < a.S; ++j) {
        const int src = j + a.L;
        const float v[1] = {src < a.S ? cv_ld1(a.st, so + src * a.sl, a.dt) : cv_ld1(a.x, xo + (int64_t)(src - a.S) * a.xl, a.dt)};
        rn_st<1>(a.st, so + j * a.sl, a.dt, v);
    }
}

// ---- host side ----------------------------------------------------------------------------------
static int cv_esize(int dt) { return dt == B200_F32 ? 4 : 2; }
static bool cv_dtype_ok(int dt) { return dt == B200_F32 || dt == B200_BF16 || dt == B200_F16; }

// widest V in {4, 2, 1} dividing C such that every base and every (batch, time) stride is aligned to V elements of its dtype
static int cv_vec(int C, int n, const void* const* ptrs, const int64_t* strides, const int* dts) {
    for (int V = 4; V > 1; V >>= 1) {
        bool ok = C % V == 0;
        for (int i = 0; i < n && ok; ++i)
            ok = reinterpret_cast<uintptr_t>(ptrs[i]) % (uintptr_t)(V * cv_esize(dts[i])) == 0 && strides[2 * i] % V == 0 &&
                 strides[2 * i + 1] % V == 0;
        if (ok) return V;
    }
    return 1;
}

static dim3 cv_grid(int32_t batch, int32_t L, int32_t C, int V) {
    return dim3((unsigned)((C + CV_THREADS * V - 1) / (CV_THREADS * V)), (unsigned)((L + CV_TL - 1) / CV_TL), (unsigned)batch);
}

static int cv_check(const char* what, int32_t batch, int32_t L, int32_t C, int32_t width) {
    B200_REQUIRE(batch >= 1 && batch <= 65535, "%s: batch = %d outside [1, 65535]", what, batch);
    B200_REQUIRE(L >= 1 && L <= 65535 * CV_TL, "%s: seqlen = %d outside [1, %d]", what, L, 65535 * CV_TL);
    B200_REQUIRE(C >= 1, "%s: dim = %d is not positive", what, C);
    B200_REQUIRE(width >= 2 && width <= 4, "%s: width = %d outside [2, 4]", what, width);
    return 0;
}

template <bool FWD, int W, int V, bool SEQ>
static int cv_launch(const ConvArgs& a, dim3 grid, cudaStream_t st) {
    if (FWD) {
        causal_conv1d_fwd_kernel<W, V, SEQ><<<grid, CV_THREADS, 0, st>>>(a);
        return check_launch("causal_conv1d_fwd_kernel");
    }
    causal_conv1d_bwd_kernel<W, V, SEQ><<<grid, CV_THREADS, 0, st>>>(a);
    return check_launch("causal_conv1d_bwd_kernel");
}

template <bool FWD, int W>
static int cv_dispatch_v(const ConvArgs& a, int V, dim3 grid, cudaStream_t st) {
    const bool seq = a.seq != nullptr;
    if (V == 4) return seq ? cv_launch<FWD, W, 4, true>(a, grid, st) : cv_launch<FWD, W, 4, false>(a, grid, st);
    if (V == 2) return seq ? cv_launch<FWD, W, 2, true>(a, grid, st) : cv_launch<FWD, W, 2, false>(a, grid, st);
    return seq ? cv_launch<FWD, W, 1, true>(a, grid, st) : cv_launch<FWD, W, 1, false>(a, grid, st);
}

template <bool FWD>
static int cv_dispatch(const ConvArgs& a, int width, int V, dim3 grid, cudaStream_t st) {
    if (width == 2) return cv_dispatch_v<FWD, 2>(a, V, grid, st);
    if (width == 3) return cv_dispatch_v<FWD, 3>(a, V, grid, st);
    return cv_dispatch_v<FWD, 4>(a, V, grid, st);
}

}  // namespace b200

using namespace b200;

extern "C" int b200_causal_conv1d_partials(int32_t batch, int32_t seqlen, int32_t dim, int32_t width) {
    if (int rc = cv_check("b200_causal_conv1d_partials", batch, seqlen, dim, width)) return rc;
    return batch * ((seqlen + CV_TL - 1) / CV_TL);
}

extern "C" int b200_causal_conv1d_fwd(const void* x, int32_t x_dtype, int64_t x_batch_stride, int64_t x_seq_stride, const float* weight,
                                      const float* bias, const int32_t* seq_idx, int64_t seq_batch_stride, int64_t seq_stride, void* out,
                                      int32_t out_dtype, int64_t out_batch_stride, int64_t out_seq_stride, int32_t batch, int32_t seqlen,
                                      int32_t dim, int32_t width, int32_t silu, b200_stream_t stream) {
    B200_REQUIRE(x && weight && out, "b200_causal_conv1d_fwd: NULL argument (x, weight and out are required)");
    if (int rc = cv_check("b200_causal_conv1d_fwd", batch, seqlen, dim, width)) return rc;
    B200_REQUIRE(cv_dtype_ok(x_dtype) && cv_dtype_ok(out_dtype), "b200_causal_conv1d_fwd: unsupported dtype x=%d out=%d", x_dtype,
                 out_dtype);
    B200_REQUIRE(x_batch_stride >= 0 && x_seq_stride >= 0 && out_batch_stride >= 0 && out_seq_stride >= 0 && seq_batch_stride >= 0 &&
                     seq_stride >= 0,
                 "b200_causal_conv1d_fwd: negative stride");
    ConvArgs a{};
    a.x = x, a.w = weight, a.b = bias, a.seq = seq_idx, a.y = out;
    a.xb = x_batch_stride, a.xl = x_seq_stride, a.sb = seq_batch_stride, a.sl = seq_stride, a.yb = out_batch_stride, a.yl = out_seq_stride;
    a.L = seqlen, a.C = dim, a.x_dt = x_dtype, a.y_dt = out_dtype, a.silu = silu != 0;
    const void* ptrs[2] = {x, out};
    const int64_t strides[4] = {x_batch_stride, x_seq_stride, out_batch_stride, out_seq_stride};
    const int dts[2] = {x_dtype, out_dtype};
    const int V = cv_vec(dim, 2, ptrs, strides, dts);
    return cv_dispatch<true>(a, width, V, cv_grid(batch, seqlen, dim, V), (cudaStream_t)stream);
}

extern "C" int b200_causal_conv1d_bwd(const float* dout, int64_t dout_batch_stride, int64_t dout_seq_stride, const void* x, int32_t x_dtype,
                                      int64_t x_batch_stride, int64_t x_seq_stride, const float* weight, const float* bias,
                                      const int32_t* seq_idx, int64_t seq_batch_stride, int64_t seq_stride, void* dx, int64_t dx_batch_stride,
                                      int64_t dx_seq_stride, float* dweight_partial, float* dbias_partial, int32_t batch, int32_t seqlen,
                                      int32_t dim, int32_t width, int32_t silu, b200_stream_t stream) {
    B200_REQUIRE(dout && x && weight && dx && dweight_partial,
                 "b200_causal_conv1d_bwd: NULL argument (dout, x, weight, dx and dweight_partial are required)");
    if (int rc = cv_check("b200_causal_conv1d_bwd", batch, seqlen, dim, width)) return rc;
    B200_REQUIRE(cv_dtype_ok(x_dtype), "b200_causal_conv1d_bwd: unsupported dtype x=%d", x_dtype);
    B200_REQUIRE(dout_batch_stride >= 0 && dout_seq_stride >= 0 && x_batch_stride >= 0 && x_seq_stride >= 0 && dx_batch_stride >= 0 &&
                     dx_seq_stride >= 0 && seq_batch_stride >= 0 && seq_stride >= 0,
                 "b200_causal_conv1d_bwd: negative stride");
    ConvArgs a{};
    a.x = x, a.w = weight, a.b = bias, a.seq = seq_idx, a.dy = dout, a.dx = dx, a.dwp = dweight_partial, a.dbp = dbias_partial;
    a.xb = x_batch_stride, a.xl = x_seq_stride, a.sb = seq_batch_stride, a.sl = seq_stride, a.gb = dout_batch_stride, a.gl = dout_seq_stride;
    a.dxb = dx_batch_stride, a.dxl = dx_seq_stride;
    a.L = seqlen, a.C = dim, a.x_dt = x_dtype, a.y_dt = x_dtype, a.silu = silu != 0;
    const void* ptrs[3] = {x, dout, dx};
    const int64_t strides[6] = {x_batch_stride, x_seq_stride, dout_batch_stride, dout_seq_stride, dx_batch_stride, dx_seq_stride};
    const int dts[3] = {x_dtype, B200_F32, x_dtype};
    const int V = cv_vec(dim, 3, ptrs, strides, dts);
    return cv_dispatch<false>(a, width, V, cv_grid(batch, seqlen, dim, V), (cudaStream_t)stream);
}

extern "C" int b200_causal_conv1d_update(const void* x, int32_t x_dtype, int64_t x_batch_stride, int64_t x_dim_stride, int64_t x_seq_stride,
                                         void* conv_state, int64_t state_batch_stride, int64_t state_dim_stride, int64_t state_seq_stride,
                                         const void* weight, int32_t weight_dtype, int64_t weight_dim_stride, int64_t weight_width_stride,
                                         const void* bias, int32_t bias_dtype, int64_t bias_stride, void* out, int64_t out_batch_stride,
                                         int64_t out_dim_stride, int64_t out_seq_stride, int32_t batch, int32_t dim, int32_t seqlen,
                                         int32_t state_len, int32_t width, int32_t silu, b200_stream_t stream) {
    B200_REQUIRE(x && conv_state && weight && out,
                 "b200_causal_conv1d_update: NULL argument (x, conv_state, weight and out are required)");
    B200_REQUIRE(batch >= 1 && batch <= 65535, "b200_causal_conv1d_update: batch = %d outside [1, 65535]", batch);
    B200_REQUIRE(seqlen >= 1, "b200_causal_conv1d_update: seqlen = %d is not positive", seqlen);
    B200_REQUIRE(dim >= 1, "b200_causal_conv1d_update: dim = %d is not positive", dim);
    B200_REQUIRE(width >= 2 && width <= 4, "b200_causal_conv1d_update: width = %d outside [2, 4]", width);
    B200_REQUIRE(state_len >= width - 1, "b200_causal_conv1d_update: state_len = %d is shorter than width - 1 = %d", state_len, width - 1);
    B200_REQUIRE(cv_dtype_ok(x_dtype) && cv_dtype_ok(weight_dtype) && (!bias || cv_dtype_ok(bias_dtype)),
                 "b200_causal_conv1d_update: unsupported dtype x=%d weight=%d bias=%d", x_dtype, weight_dtype, bias_dtype);
    B200_REQUIRE(x_batch_stride >= 0 && x_dim_stride >= 0 && x_seq_stride >= 0 && state_batch_stride >= 0 && state_dim_stride >= 0 &&
                     state_seq_stride >= 0 && weight_dim_stride >= 0 && weight_width_stride >= 0 && bias_stride >= 0 &&
                     out_batch_stride >= 0 && out_dim_stride >= 0 && out_seq_stride >= 0,
                 "b200_causal_conv1d_update: negative stride");
    ConvUpdateArgs a{};
    a.x = x, a.st = conv_state, a.w = weight, a.b = bias, a.y = out;
    a.xb = x_batch_stride, a.xc = x_dim_stride, a.xl = x_seq_stride, a.sb = state_batch_stride, a.sc = state_dim_stride;
    a.sl = state_seq_stride, a.wc = weight_dim_stride, a.wk = weight_width_stride, a.bs = bias_stride;
    a.yb = out_batch_stride, a.yc = out_dim_stride, a.yl = out_seq_stride;
    a.C = dim, a.L = seqlen, a.S = state_len, a.dt = x_dtype, a.w_dt = weight_dtype, a.b_dt = bias_dtype, a.silu = silu != 0;
    const dim3 grid((unsigned)((dim + CV_THREADS - 1) / CV_THREADS), (unsigned)batch);
    const cudaStream_t st = (cudaStream_t)stream;
    if (width == 2) causal_conv1d_update_kernel<2><<<grid, CV_THREADS, 0, st>>>(a);
    else if (width == 3) causal_conv1d_update_kernel<3><<<grid, CV_THREADS, 0, st>>>(a);
    else causal_conv1d_update_kernel<4><<<grid, CV_THREADS, 0, st>>>(a);
    return check_launch("causal_conv1d_update_kernel");
}
