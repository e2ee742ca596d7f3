// state_update.cu -- one recurrent step of a Mamba state (mamba_ssm 2.2.2's selective_state_update), sm_100a.
//
// For every (batch b, head h, row p of the head) and n < dstate, all arithmetic fp32, g = h / (nheads / ngroups):
//
//   dt' = softplus20?(dt[b,h,p] + dt_bias[h,p])        state[b,h,p,n] <- state * exp(A[h,p,n] dt') + (B[b,g,n] dt') x[b,h,p]
//   out[b,h,p] = (sum_n state'[n] C[b,g,n] + D[h,p] x[b,h,p]) * silu?(z[b,h,p])
//
// with the fp32 updated state state' (before it is rounded to the state's dtype) in the sum.  The cost is bandwidth: the state is
// read and written once per call.  Layout: CTA = (tile of head rows, head, batch row), 128 threads.  A row of dstate elements is
// owned by `lpr` lanes (a power of two <= 32, the fewest that cover dstate / V vectors), each holding up to 8 / V vectors of V
// consecutive state elements; the row's dot product with C is a shuffle reduction over those lanes.  Each lane loads the B and C
// elements of its own vectors once into registers and keeps them for every row it visits (no shared memory, no barrier).  The
// state is streamed with the widest vector its base and strides allow, and the loads of SSU_R rows are issued before their
// arithmetic.  When A, dt and dt_bias have stride 0 over (p, n) -- transformers' expanded Mamba-2 arguments -- exp(A dt') is
// formed once per thread instead of once per element.  Every other tensor is read through its strides in its own dtype.
#include "common.cuh"

namespace b200 {

constexpr int SSU_THREADS = 128;
constexpr int SSU_R = 4;          // rows per row group whose state loads are issued together
constexpr int SSU_MAX_DSTATE = 256;

// one element of a f32 / bf16 / f16 tensor that no kernel writes
__device__ __forceinline__ float ssu_ld(const void* base, int64_t idx, int dt) {
    if (dt == B200_F32) return __ldg(static_cast<const float*>(base) + idx);
    const unsigned short h = __ldg(static_cast<const unsigned short*>(base) + idx);
    return dt == B200_BF16 ? __uint_as_float((uint32_t)h << 16) : __half2float(__ushort_as_half(h));
}

__device__ __forceinline__ float ssu_dt(const b200_ssu_params& p, int64_t b, int h, int row) {
    float v = ssu_ld(p.dt, b * p.dt_stride[0] + h * p.dt_stride[1] + row * p.dt_stride[2], p.dt_dtype);
    if (p.dt_bias) v += ssu_ld(p.dt_bias, h * p.dt_bias_stride[0] + row * p.dt_bias_stride[1], p.dt_bias_dtype);
    return p.dt_softplus ? softplus20(v) : v;
}

// V consecutive state elements (V > 1: unit n stride) per vector, K vectors per lane: K = 1 when 32 lanes cover dstate, else
// 8 / V, which covers dstate <= 256
template <int V, int K>
__global__ void __launch_bounds__(SSU_THREADS) ssu_kernel(const b200_ssu_params p, const int lpr, const int rows_per_cta, const int tied) {
    const int lr = threadIdx.x & (lpr - 1);
    const int rg = threadIdx.x / lpr, ngr = SSU_THREADS / lpr;
    const int h = blockIdx.y;
    const int64_t b = blockIdx.z;
    const int g = h / (p.nheads / p.ngroups);
    const int pbeg = blockIdx.x * rows_per_cta, pend = min(pbeg + rows_per_cta, p.headdim);
    float Bv[K][V], Cv[K][V];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int n0 = (lr + k * lpr) * V;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const bool ok = n0 + j < p.dstate;
            Bv[k][j] = ok ? ssu_ld(p.B, b * p.B_stride[0] + g * p.B_stride[1] + (n0 + j) * p.B_stride[2], p.B_dtype) : 0.f;
            Cv[k][j] = ok ? ssu_ld(p.C, b * p.C_stride[0] + g * p.C_stride[1] + (n0 + j) * p.C_stride[2], p.C_dtype) : 0.f;
        }
    }
    float dt_tied = 0.f, dA_tied = 0.f;
    if (tied) {
        dt_tied = ssu_dt(p, b, h, 0);
        dA_tied = exp_acc(ssu_ld(p.A, h * p.A_stride[0], p.A_dtype) * dt_tied);
    }
    const int64_t sbase = b * p.state_stride[0] + h * p.state_stride[1];
    // the trip count is the same for every lane of the CTA: the shuffles below run with all lanes present
    for (int pb = pbeg; pb < pend; pb += ngr * SSU_R) {
        uint32_t r[SSU_R][K][V];
#pragma unroll
        for (int u = 0; u < SSU_R; ++u) {
            const int row = pb + u * ngr + rg;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int n0 = (lr + k * lpr) * V;
                if (row < pend && n0 < p.dstate)
                    rn_ld<V>(p.state, sbase + row * p.state_stride[2] + n0 * p.state_stride[3], p.state_dtype, r[u][k]);
            }
        }
#pragma unroll
        for (int u = 0; u < SSU_R; ++u) {
            const int row = pb + u * ngr + rg;
            const bool live = row < pend;
            float acc = 0.f, xv = 0.f;
            if (live) {
                xv = ssu_ld(p.x, b * p.x_stride[0] + h * p.x_stride[1] + row * p.x_stride[2], p.x_dtype);
                const float dtv = tied ? dt_tied : ssu_dt(p, b, h, row);
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int n0 = (lr + k * lpr) * V;
                    if (n0 < p.dstate) {
                        float s[V];
                        rn_cvt<V>(r[u][k], p.state_dtype, s);
#pragma unroll
                        for (int j = 0; j < V; ++j) {
                            const float dA = tied ? dA_tied
                                                  : exp_acc(ssu_ld(p.A, h * p.A_stride[0] + row * p.A_stride[1] + (n0 + j) * p.A_stride[2],
                                                                   p.A_dtype) * dtv);
                            s[j] = fmaf(s[j], dA, Bv[k][j] * dtv * xv);
                            acc = fmaf(s[j], Cv[k][j], acc);
                        }
                        rn_st<V>(p.state, sbase + row * p.state_stride[2] + n0 * p.state_stride[3], p.state_dtype, s);
                    }
                }
            }
            for (int off = lpr >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if (live && lr == 0) {
                if (p.D) acc = fmaf(ssu_ld(p.D, h * p.D_stride[0] + row * p.D_stride[1], p.D_dtype), xv, acc);
                if (p.z) {
                    const float zv = ssu_ld(p.z, b * p.z_stride[0] + h * p.z_stride[1] + row * p.z_stride[2], p.z_dtype);
                    acc *= zv * sigmoidf_(zv);
                }
                rn_st<1>(p.out, b * p.out_stride[0] + h * p.out_stride[1] + row * p.out_stride[2], p.out_dtype, &acc);
            }
        }
    }
}

static bool ssu_dtype_ok(int dt) { return dt == B200_F32 || dt == B200_BF16 || dt == B200_F16; }

template <int N>
static bool ssu_nonneg(const int64_t (&s)[N]) {
    for (int i = 0; i < N; ++i)
        if (s[i] < 0) return false;
    return true;
}

}  // namespace b200

using namespace b200;

extern "C" int b200_selective_state_update(const b200_ssu_params* p, b200_stream_t stream) {
    B200_REQUIRE(p, "b200_selective_state_update: NULL params");
    const b200_ssu_params& q = *p;
    B200_REQUIRE(q.batch >= 1 && q.batch <= 65535, "b200_selective_state_update: batch = %d outside [1, 65535]", q.batch);
    B200_REQUIRE(q.nheads >= 1 && q.nheads <= 65535, "b200_selective_state_update: nheads = %d outside [1, 65535]", q.nheads);
    B200_REQUIRE(q.headdim >= 1, "b200_selective_state_update: headdim = %d is not positive", q.headdim);
    B200_REQUIRE(q.ngroups >= 1 && q.nheads % q.ngroups == 0, "b200_selective_state_update: nheads = %d is not a multiple of ngroups = %d",
                 q.nheads, q.ngroups);
    B200_REQUIRE(q.dstate >= 1 && q.dstate <= SSU_MAX_DSTATE, "b200_selective_state_update: dstate = %d outside [1, %d]", q.dstate,
                 SSU_MAX_DSTATE);
    B200_REQUIRE(q.state && q.x && q.dt && q.A && q.B && q.C && q.out,
                 "b200_selective_state_update: NULL argument (state, x, dt, A, B, C and out are required)");
    const int dts[10] = {q.state_dtype, q.x_dtype, q.dt_dtype, q.A_dtype, q.B_dtype, q.C_dtype, q.out_dtype,
                         q.D ? q.D_dtype : 0, q.z ? q.z_dtype : 0, q.dt_bias ? q.dt_bias_dtype : 0};
    for (int i = 0; i < 10; ++i)
        B200_REQUIRE(ssu_dtype_ok(dts[i]), "b200_selective_state_update: unsupported dtype code %d (argument %d)", dts[i], i);
    B200_REQUIRE(ssu_nonneg(q.state_stride) && ssu_nonneg(q.x_stride) && ssu_nonneg(q.dt_stride) && ssu_nonneg(q.A_stride) &&
                     ssu_nonneg(q.B_stride) && ssu_nonneg(q.C_stride) && ssu_nonneg(q.D_stride) && ssu_nonneg(q.z_stride) &&
                     ssu_nonneg(q.dt_bias_stride) && ssu_nonneg(q.out_stride),
                 "b200_selective_state_update: negative stride");
    // V: the widest vector every state base and (batch, head, row) stride allows, with unit stride along dstate
    const int es = q.state_dtype == B200_F32 ? 4 : 2;
    int V = 1;
    for (int v = 4; v > 1 && V == 1; v >>= 1)
        if (q.dstate % v == 0 && q.state_stride[3] == 1 && reinterpret_cast<uintptr_t>(q.state) % (uintptr_t)(v * es) == 0 &&
            q.state_stride[0] % v == 0 && q.state_stride[1] % v == 0 && q.state_stride[2] % v == 0)
            V = v;
    const int nvec = q.dstate / V;
    int lpr = 1;
    while (lpr < 32 && lpr < nvec) lpr <<= 1;
    const int tied = q.A_stride[1] == 0 && q.A_stride[2] == 0 && q.dt_stride[2] == 0 && (!q.dt_bias || q.dt_bias_stride[1] == 0);
    // rows per CTA: up to 4 passes of every row group, fewer while the grid would not give each of the 148 SMs 4 CTAs
    const int pass_rows = SSU_THREADS / lpr * SSU_R;
    int passes = 4;
    while (passes > 1 && (int64_t)((q.headdim + pass_rows * passes - 1) / (pass_rows * passes)) * q.nheads * q.batch < 4 * 148) passes >>= 1;
    const int rows = pass_rows * passes;
    const dim3 grid((unsigned)((q.headdim + rows - 1) / rows), (unsigned)q.nheads, (unsigned)q.batch);
    const cudaStream_t st = (cudaStream_t)stream;
    const bool k1 = nvec <= 32;
    if (V == 4) k1 ? ssu_kernel<4, 1><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied) : ssu_kernel<4, 2><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied);
    else if (V == 2) k1 ? ssu_kernel<2, 1><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied) : ssu_kernel<2, 4><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied);
    else k1 ? ssu_kernel<1, 1><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied) : ssu_kernel<1, 8><<<grid, SSU_THREADS, 0, st>>>(q, lpr, rows, tied);
    return check_launch("ssu_kernel");
}
