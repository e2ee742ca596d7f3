// rmsnorm.cu -- gated RMSNorm with groups, forward and backward, sm_100a.
//
// The semantics of mamba_ssm's layernorm_gated.rms_norm_ref (mamba_ssm 2.2.2), which SS2D_with_SSD (reference
// SSD/MedSSD.py:268-269, 393-394) and CrossMamba build through RMSNorm(d_ssm, norm_before_gate, group_size = d_ssm / ngroups).
// A row of `dim` columns is cut into dim / gs contiguous groups, each normalised on its own, all arithmetic in fp32:
//
//   norm_before_gate = 0:  out = rmsnorm_g(x * silu(z)) * w [+ b]
//   norm_before_gate = 1:  out = (rmsnorm_g(x) * w [+ b]) * silu(z)
//   z == NULL:             out = rmsnorm_g(x) * w [+ b]            rmsnorm_g(v) = v * rsqrt(mean_group(v^2) + eps)
//
// Backward, with v the normalised input (x * silu(z) before the gate, x otherwise), nh = v * rstd, gate = silu(z) after the norm
// (1 otherwise):
//   du = dy * gate        dw += du * nh        db += du        dn = du * w
//   dv = rstd * (dn - nh * mean_group(dn * nh));   dx = dv [* silu(z) before the gate]
//   dz = dv * x * silu'(z) (before the gate) or dy * (nh * w + b) * silu'(z) (after it)
//
// Layout: CTA (bx, g) handles group g of rows bx*TPC + team, stepping gridDim.x * TPC, where a team of T threads (one warp for
// groups of up to 1024 columns, the whole CTA up to 8192) holds one group of one row in registers: NPL values per thread, as
// NPL / V vectors of V consecutive columns.  A team always sees the same group, so d(weight) / d(bias) accumulate in registers
// over the team's rows and the CTA writes them as one partial row (no atomics: the same grid gives the same sums).  x, z and dy are
// read in place with their own dtype and row stride (z is a column slice of in_proj's output); V is the widest vector that every
// tensor's base, row stride and group offset allow, 1 when one of them is only element-aligned.  One read of x / z (/ dy) and one
// write of each output per element.  MedSSD under bf16 autocast (fp32 x from the cross-merge, bf16 z, bf16 out and dy) moves
// 4 + 2 + 2 = 8 B forward and 2 + 4 + 2 + 4 + 2 = 14 B backward (dy, x, z in; dx, dz out) per element.
#include "common.cuh"

namespace b200 {

constexpr int RN_THREADS = 256;
constexpr int RN_MAXDIM = 8192;          // 32 columns per thread of a 256-thread team
constexpr int RN_CTAS = 148 * 8;         // 2048 threads per SM

__device__ __forceinline__ float rn_silu(float z) { return z / (1.f + expf(-z)); }

// V consecutive elements as raw bits: the loads of a row are all issued before the first conversion (rn_cvt)
template <int V>
__device__ __forceinline__ void rn_ld(const void* base, int64_t idx, int dt, uint32_t (&r)[V]) {
    if (dt == B200_F32) {
        const float* p = static_cast<const float*>(base) + idx;
        if constexpr (V == 4) {
            const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
            r[0] = u.x, r[1] = u.y, r[2] = u.z, r[3] = u.w;
        } else if constexpr (V == 2) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p));
            r[0] = u.x, r[1] = u.y;
        } else {
            r[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
        }
    } else {
        const unsigned short* p = static_cast<const unsigned short*>(base) + idx;
        if constexpr (V == 4) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p));
            r[0] = u.x, r[1] = u.y;
        } else if constexpr (V == 2) {
            r[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
        } else {
            r[0] = __ldcs(p);
        }
    }
}

template <int V>
__device__ __forceinline__ void rn_cvt(const uint32_t (&r)[V], int dt, float* v) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        if (dt == B200_F32) {
            v[j] = __uint_as_float(r[j]);
        } else {
            const uint32_t h = V == 1 ? r[0] & 0xffffu : (r[j >> 1] >> (16 * (j & 1))) & 0xffffu;
            v[j] = dt == B200_BF16 ? __uint_as_float(h << 16) : __half2float(__ushort_as_half((unsigned short)h));
        }
    }
}

template <int V>
__device__ __forceinline__ void rn_st(void* base, int64_t idx, int dt, const float* v) {
    if (dt == B200_F32) {
        float* p = static_cast<float*>(base) + idx;
        if constexpr (V == 4) __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
        else if constexpr (V == 2) __stcs(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
        else __stcs(p, v[0]);
        return;
    }
    uint32_t h[V];
#pragma unroll
    for (int j = 0; j < V; ++j)
        h[j] = dt == B200_BF16 ? __bfloat16_as_ushort(__float2bfloat16_rn(v[j])) : __half_as_ushort(__float2half_rn(v[j]));
    unsigned short* p = static_cast<unsigned short*>(base) + idx;
    if constexpr (V == 4) __stcs(reinterpret_cast<uint2*>(p), make_uint2(h[0] | h[1] << 16, h[2] | h[3] << 16));
    else if constexpr (V == 2) __stcs(reinterpret_cast<unsigned int*>(p), h[0] | h[1] << 16);
    else __stcs(p, (unsigned short)h[0]);
}

// sum over a team: a warp, or the whole CTA (then every thread of the CTA calls it at the same point)
template <int T>
__device__ __forceinline__ float rn_team_sum(float v, float* sbuf) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if constexpr (T == 32) {
        return v;
    } else {
        static_assert(T == RN_THREADS, "a team is one warp or the whole CTA");
        __syncthreads();   // the previous call's readers are done with sbuf
        if ((threadIdx.x & 31) == 0) sbuf[threadIdx.x >> 5] = v;
        __syncthreads();
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < RN_THREADS / 32; ++i) s += sbuf[i];
        return s;
    }
}

struct RmsFwdArgs {
    const void* x;
    const void* z;
    const float* w;
    const float* b;
    void* out;
    float* rstd;
    int64_t xs, zs, rows;
    int dim, gs, x_dt, z_dt, out_dt, nbg;
    float eps;
};

struct RmsBwdArgs {
    const void* dy;
    const void* x;
    const void* z;
    const float* w;
    const float* b;
    const float* rstd;
    void* dx;
    void* dz;
    float* dwp;
    float* dbp;
    int64_t dys, xs, zs, rows;
    int dim, gs, dy_dt, x_dt, z_dt, nbg;
};

template <int T, int NPL, int V>
__global__ void __launch_bounds__(RN_THREADS) rmsnorm_fwd_kernel(const RmsFwdArgs a) {
    constexpr int TPC = RN_THREADS / T, KV = NPL / V;
    __shared__ float sbuf[RN_THREADS / 32];
    const int t = threadIdx.x % T, team = threadIdx.x / T;
    const int g = blockIdx.y;
    const int64_t c0 = (int64_t)g * a.gs;
    const bool hz = a.z != nullptr, gate_in = hz && !a.nbg, gate_out = hz && a.nbg;
    for (int64_t r = (int64_t)blockIdx.x * TPC + team; r < a.rows; r += (int64_t)gridDim.x * TPC) {
        uint32_t rx[KV][V], rz[KV][V];
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                rn_ld<V>(a.x, r * a.xs + c0 + c, a.x_dt, rx[k]);
                if (hz) rn_ld<V>(a.z, r * a.zs + c0 + c, a.z_dt, rz[k]);
            }
        }
        float v[NPL], zv[NPL];
        float ss = 0.f;
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                rn_cvt<V>(rx[k], a.x_dt, v + k * V);
                if (hz) rn_cvt<V>(rz[k], a.z_dt, zv + k * V);
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    if (gate_in) v[k * V + j] *= rn_silu(zv[k * V + j]);
                    ss += v[k * V + j] * v[k * V + j];
                }
            }
        }
        const float rs = rsqrtf(rn_team_sum<T>(ss, sbuf) / (float)a.gs + a.eps);
        if (t == 0) a.rstd[r * gridDim.y + g] = rs;
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                float o[V];
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    o[j] = v[k * V + j] * rs * __ldg(a.w + c0 + c + j);
                    if (a.b) o[j] += __ldg(a.b + c0 + c + j);
                    if (gate_out) o[j] *= rn_silu(zv[k * V + j]);
                }
                rn_st<V>(a.out, r * a.dim + c0 + c, a.out_dt, o);
            }
        }
    }
}

template <int T, int NPL, int V>
__global__ void __launch_bounds__(RN_THREADS) rmsnorm_bwd_kernel(const RmsBwdArgs a) {
    constexpr int TPC = RN_THREADS / T, KV = NPL / V;
    __shared__ float sbuf[RN_THREADS / 32];
    __shared__ float red[TPC][T * NPL];
    const int t = threadIdx.x % T, team = threadIdx.x / T;
    const int g = blockIdx.y;
    const int64_t c0 = (int64_t)g * a.gs;
    const bool hz = a.z != nullptr, gate_in = hz && !a.nbg, gate_out = hz && a.nbg;
    float aw[NPL], ab[NPL];
#pragma unroll
    for (int i = 0; i < NPL; ++i) aw[i] = ab[i] = 0.f;
    for (int64_t r = (int64_t)blockIdx.x * TPC + team; r < a.rows; r += (int64_t)gridDim.x * TPC) {
        uint32_t rg[KV][V], rx[KV][V], rz[KV][V];
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                rn_ld<V>(a.dy, r * a.dys + c0 + c, a.dy_dt, rg[k]);
                rn_ld<V>(a.x, r * a.xs + c0 + c, a.x_dt, rx[k]);
                if (hz) rn_ld<V>(a.z, r * a.zs + c0 + c, a.z_dt, rz[k]);
            }
        }
        const float rs = __ldg(a.rstd + r * gridDim.y + g);
        float dn[NPL], xv[NPL], zv[NPL];   // dy -> du * w
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                rn_cvt<V>(rg[k], a.dy_dt, dn + k * V);
                rn_cvt<V>(rx[k], a.x_dt, xv + k * V);
                if (hz) rn_cvt<V>(rz[k], a.z_dt, zv + k * V);
                float dzo[V];
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int i = k * V + j;
                    const float wc = __ldg(a.w + c0 + c + j);
                    float vv = xv[i], du = dn[i];
                    if (hz) {
                        const float zz = zv[i], sg = 1.f / (1.f + expf(-zz)), sl = zz * sg;
                        if (gate_in) vv *= sl;
                        if (gate_out) {
                            const float u = vv * rs * wc + (a.b ? __ldg(a.b + c0 + c + j) : 0.f);
                            dzo[j] = du * u * sg * (1.f + zz * (1.f - sg));
                            du *= sl;
                        }
                    }
                    const float nh = vv * rs;
                    aw[i] += du * nh;
                    ab[i] += du;
                    dn[i] = du * wc;
                    s += dn[i] * nh;
                }
                if (gate_out) rn_st<V>(a.dz, r * a.dim + c0 + c, a.z_dt, dzo);
            }
        }
        const float m = rn_team_sum<T>(s, sbuf) / (float)a.gs;
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
            if (c < a.gs) {
                float dxo[V], dzo[V];
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int i = k * V + j;
                    if (gate_in) {
                        const float zz = zv[i], sg = 1.f / (1.f + expf(-zz)), sl = zz * sg;
                        const float dv = rs * (dn[i] - xv[i] * sl * rs * m);
                        dxo[j] = dv * sl;
                        dzo[j] = dv * xv[i] * sg * (1.f + zz * (1.f - sg));
                    } else {
                        dxo[j] = rs * (dn[i] - xv[i] * rs * m);
                    }
                }
                rn_st<V>(a.dx, r * a.dim + c0 + c, a.x_dt, dxo);
                if (gate_in) rn_st<V>(a.dz, r * a.dim + c0 + c, a.z_dt, dzo);
            }
        }
    }
    // d(weight), d(bias): the CTA's teams (all on group g) are combined in a fixed order into one partial row per CTA
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        float* part = pass ? a.dbp : a.dwp;
        if (part == nullptr) break;
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            const int c = (t + T * k) * V;
#pragma unroll
            for (int j = 0; j < V; ++j)
                if (c < a.gs) red[team][c + j] = pass ? ab[k * V + j] : aw[k * V + j];
        }
        __syncthreads();
        for (int c = threadIdx.x; c < a.gs; c += RN_THREADS) {
            float acc = 0.f;
#pragma unroll
            for (int tm = 0; tm < TPC; ++tm) acc += red[tm][c];
            part[(int64_t)blockIdx.x * a.dim + c0 + c] = acc;
        }
        __syncthreads();
    }
}

// ---- host side ----------------------------------------------------------------------------------
static int rn_team(int gs) { return gs <= 1024 ? 32 : RN_THREADS; }

static int rn_grid_x(int64_t rows, int dim, int gs) {
    const int tpc = RN_THREADS / rn_team(gs), ngroups = dim / gs;
    const int64_t by_rows = (rows + tpc - 1) / tpc, by_sms = (RN_CTAS + ngroups - 1) / ngroups;
    const int64_t gx = by_rows < by_sms ? by_rows : by_sms;
    return (int)(gx < 1 ? 1 : gx);
}

static int rn_esize(int dt) { return dt == B200_F32 ? 4 : 2; }

// widest V in {4, 2, 1} such that every (base, row stride) pair is aligned to V elements of its dtype and gs % V == 0
static int rn_vec(int gs, int n, const void* const* ptrs, const int64_t* strides, const int* dts) {
    for (int V = 4; V > 1; V >>= 1) {
        bool ok = gs % V == 0;
        for (int i = 0; i < n && ok; ++i)
            ok = ptrs[i] == nullptr || (reinterpret_cast<uintptr_t>(ptrs[i]) % (uintptr_t)(V * rn_esize(dts[i])) == 0 && strides[i] % V == 0);
        if (ok) return V;
    }
    return 1;
}

template <int T, int NPL, int V>
static int rn_launch_fwd(const RmsFwdArgs& a, dim3 grid, cudaStream_t st) {
    rmsnorm_fwd_kernel<T, NPL, V><<<grid, RN_THREADS, 0, st>>>(a);
    return check_launch("rmsnorm_fwd_kernel");
}
template <int T, int NPL, int V>
static int rn_launch_bwd(const RmsBwdArgs& a, dim3 grid, cudaStream_t st) {
    rmsnorm_bwd_kernel<T, NPL, V><<<grid, RN_THREADS, 0, st>>>(a);
    return check_launch("rmsnorm_bwd_kernel");
}

// (team, columns per thread, vector width) from the group size and V: the smallest register row that holds a group
#define RN_DISPATCH(FN, gs, V, ...)                                                            \
    do {                                                                                       \
        const int T_ = rn_team(gs), npl_ = (gs + T_ - 1) / T_;                                  \
        if (T_ == 32) {                                                                        \
            if (npl_ <= 4) RN_VEC(FN, 32, 4, V, __VA_ARGS__);                                   \
            if (npl_ <= 8) RN_VEC(FN, 32, 8, V, __VA_ARGS__);                                   \
            if (npl_ <= 16) RN_VEC(FN, 32, 16, V, __VA_ARGS__);                                 \
            RN_VEC(FN, 32, 32, V, __VA_ARGS__);                                                 \
        }                                                                                      \
        if (npl_ <= 8) RN_VEC(FN, RN_THREADS, 8, V, __VA_ARGS__);                               \
        if (npl_ <= 16) RN_VEC(FN, RN_THREADS, 16, V, __VA_ARGS__);                             \
        RN_VEC(FN, RN_THREADS, 32, V, __VA_ARGS__);                                             \
    } while (0)
#define RN_VEC(FN, T, NPL, V, ...)                                \
    do {                                                          \
        if ((V) == 4) return FN<T, NPL, 4>(__VA_ARGS__);          \
        if ((V) == 2) return FN<T, NPL, 2>(__VA_ARGS__);          \
        return FN<T, NPL, 1>(__VA_ARGS__);                        \
    } while (0)

static int rn_check_shape(const char* what, int64_t rows, int32_t dim, int32_t gs) {
    B200_REQUIRE(rows >= 0, "%s: rows = %lld is negative", what, (long long)rows);
    B200_REQUIRE(dim >= 1 && dim <= RN_MAXDIM, "%s: dim = %d outside [1, %d]", what, dim, RN_MAXDIM);
    B200_REQUIRE(gs >= 1 && dim % gs == 0, "%s: group_size = %d does not divide dim = %d", what, gs, dim);
    return 0;
}

static bool rn_dtype_ok(int dt) { return dt == B200_F32 || dt == B200_BF16 || dt == B200_F16; }

}  // namespace b200

using namespace b200;

extern "C" int b200_rmsnorm_grid(int64_t rows, int32_t dim, int32_t group_size) {
    if (int rc = rn_check_shape("b200_rmsnorm_grid", rows, dim, group_size)) return rc;
    return rn_grid_x(rows, dim, group_size);
}

extern "C" int b200_rmsnorm_fwd(const void* x, int32_t x_dtype, int64_t x_row_stride, const void* z, int32_t z_dtype, int64_t z_row_stride,
                                const float* w, const float* b, void* out, int32_t out_dtype, float* rstd, int64_t rows, int32_t dim,
                                int32_t group_size, int32_t norm_before_gate, float eps, b200_stream_t stream) {
    B200_REQUIRE(x && w && out && rstd, "b200_rmsnorm_fwd: NULL argument (x, w, out and rstd are required)");
    if (int rc = rn_check_shape("b200_rmsnorm_fwd", rows, dim, group_size)) return rc;
    B200_REQUIRE(rn_dtype_ok(x_dtype) && rn_dtype_ok(out_dtype) && (!z || rn_dtype_ok(z_dtype)),
                 "b200_rmsnorm_fwd: unsupported dtype x=%d z=%d out=%d", x_dtype, z_dtype, out_dtype);
    B200_REQUIRE(x_row_stride >= 0 && z_row_stride >= 0, "b200_rmsnorm_fwd: negative row stride");
    if (rows == 0) return 0;
    const RmsFwdArgs a{x, z, w, b, out, rstd, x_row_stride, z_row_stride, rows, dim, group_size, x_dtype, z ? z_dtype : B200_F32,
                       out_dtype, norm_before_gate != 0, eps};
    const void* ptrs[3] = {x, z, out};
    const int64_t strides[3] = {x_row_stride, z_row_stride, dim};
    const int dts[3] = {a.x_dt, a.z_dt, out_dtype};
    const int V = rn_vec(group_size, 3, ptrs, strides, dts);
    const dim3 grid((unsigned)rn_grid_x(rows, dim, group_size), (unsigned)(dim / group_size));
    RN_DISPATCH(rn_launch_fwd, group_size, V, a, grid, (cudaStream_t)stream);
}

extern "C" int b200_rmsnorm_bwd(const void* dy, int32_t dy_dtype, int64_t dy_row_stride, const void* x, int32_t x_dtype, int64_t x_row_stride,
                                const void* z, int32_t z_dtype, int64_t z_row_stride, const float* w, const float* b, const float* rstd,
                                void* dx, void* dz, float* dw_partial, float* db_partial, int64_t rows, int32_t dim, int32_t group_size,
                                int32_t norm_before_gate, b200_stream_t stream) {
    B200_REQUIRE(dy && x && w && rstd && dx && dw_partial, "b200_rmsnorm_bwd: NULL argument (dy, x, w, rstd, dx and dw_partial are required)");
    B200_REQUIRE((z == nullptr) == (dz == nullptr), "b200_rmsnorm_bwd: dz must be given exactly when z is");
    if (int rc = rn_check_shape("b200_rmsnorm_bwd", rows, dim, group_size)) return rc;
    B200_REQUIRE(rn_dtype_ok(dy_dtype) && rn_dtype_ok(x_dtype) && (!z || rn_dtype_ok(z_dtype)),
                 "b200_rmsnorm_bwd: unsupported dtype dy=%d x=%d z=%d", dy_dtype, x_dtype, z_dtype);
    B200_REQUIRE(dy_row_stride >= 0 && x_row_stride >= 0 && z_row_stride >= 0, "b200_rmsnorm_bwd: negative row stride");
    const RmsBwdArgs a{dy, x, z, w, b, rstd, dx, dz, dw_partial, db_partial, dy_row_stride, x_row_stride, z_row_stride, rows, dim, group_size,
                       dy_dtype, x_dtype, z ? z_dtype : B200_F32, norm_before_gate != 0};
    const void* ptrs[5] = {dy, x, z, dx, dz};
    const int64_t strides[5] = {dy_row_stride, x_row_stride, z_row_stride, dim, dim};
    const int dts[5] = {dy_dtype, x_dtype, a.z_dt, x_dtype, a.z_dt};
    const int V = rn_vec(group_size, 5, ptrs, strides, dts);
    // rows == 0 still launches: the partials are written (as zeros) whatever the row count
    const dim3 grid((unsigned)rn_grid_x(rows, dim, group_size), (unsigned)(dim / group_size));
    RN_DISPATCH(rn_launch_bwd, group_size, V, a, grid, (cudaStream_t)stream);
}
