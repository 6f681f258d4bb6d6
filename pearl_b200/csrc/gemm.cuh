// gemm.cuh — the one tiled fp32 contraction kernel the actor-critic learners (sac.cu, ppo.cu) are built from.
//   C[i][j] = sum_c A(i, c) * B(j, c)        i < Mo, j < No, c < Kc
// covers nn.Linear forward (y = act(x W^T + b)), backward-data (dx = dy W, optionally masked by the ReLU of
// the layer below and accumulated) and backward-weight (dW = dy^T x, the bias gradient as an implicit
// ones column of x).  Operands are described by `Mat`: a row-major matrix whose feature axis may be the
// concatenation of two sources (state || action) and, per blockIdx.z, one of several stacked networks
// (twin critics).  Which Mat axis is the output index and which the contraction index is a template
// parameter, so the global loads are coalesced along the contiguous axis in every mode.
// fp32 FMA in a fixed order (deterministic); the next chunk's operands are prefetched into registers
// while the current chunk is multiplied.
#pragma once
#include <string.h>

#include "common.cuh"

namespace prl {

struct Mat {
    const float *p1; int ld1; int split;   // features [0, split) from p1
    const float *p2; int ld2;              // features [split, ..) from p2
    int ones_at;                           // feature index that reads as 1.0 (-1: none)
    long long net_stride1, net_stride2;    // added per blockIdx.z
    // branch-free address (selects only), so that a thread's loads of one chunk are all in flight together
    __device__ __forceinline__ const float *addr(int row, int f, int z) const {
        const float *a = p1 + z * net_stride1 + (size_t)row * ld1 + f;
        const float *b = p2 + z * net_stride2 + (size_t)row * ld2 + (f - split);
        return f < split ? a : b;
    }
};
inline Mat mat(const float *p, int ld, long long net_stride = 0) {
    Mat m; m.p1 = p; m.ld1 = ld; m.split = 1 << 30; m.p2 = nullptr; m.ld2 = 0; m.ones_at = -1; m.net_stride1 = net_stride; m.net_stride2 = 0;
    return m;
}
inline Mat mat2(const float *p1, int ld1, int split, const float *p2, int ld2, long long s1 = 0, long long s2 = 0) {
    Mat m = mat(p1, ld1, s1); m.split = split; m.p2 = p2; m.ld2 = ld2; m.net_stride2 = s2;
    return m;
}

struct GemmArgs {
    Mat A, B;
    int Mo, No, Kc;
    float *C; int ldc; long long c_net_stride;
    float *C_tail; int tail_col; long long tail_net_stride;   // column tail_col of C goes to C_tail[z][row] (bias gradient)
    const float *bias; long long bias_net_stride;             // + bias[j]
    int relu;                                                   // max(., 0)
    const float *mask; int ldm; long long mask_net_stride;     // keep only where mask[i][j] > 0
    int accumulate;                                             // C += (before relu / mask)
    long long *stamps;                                          // developer profiling of k_gemm_tc (CTA 0): [chunk][8] SM clocks
};

constexpr int GK = 32;   // contraction chunk

// AO / BO: true = the Mat's ROW index is the output index (features are contracted); false = rows are contracted
// MR x 4 outputs per thread: MR = 4 for the big tiles, MR = 2 doubles the warps of the small (latency-bound) tiles.
// KS > 1 ("slice-K"): KS groups of NT threads walk interleaved chunks of the contraction axis of the SAME tile and their
// partial sums are added in a fixed order through shared memory.  The learners' small products (batch 256-512, widths
// 64-256) fill one CTA per SM at most and a CTA's chunk loop is a chain of global-load latencies; KS = 4 puts four such
// chains on the SM at once without any global workspace.
__device__ __forceinline__ void gemm_emit(const GemmArgs &g, int z, int i, int j, float v) {
    if (g.C_tail && j == g.tail_col) { g.C_tail[z * g.tail_net_stride + i] = v; return; }
    float *dst = g.C + z * g.c_net_stride + (size_t)i * g.ldc + j;
    if (g.bias) v += __ldg(g.bias + z * g.bias_net_stride + j);
    if (g.accumulate) v += *dst;
    if (g.relu) v = fmaxf(v, 0.f);
    if (g.mask && !(__ldg(g.mask + z * g.mask_net_stride + (size_t)i * g.ldm + j) > 0.f)) v = 0.f;
    *dst = v;
}

template <int TM, int TN, int MR, int KS, bool AO, bool BO>
__global__ void __launch_bounds__((TM / MR) * (TN / 4) * KS) k_gemm(const GemmArgs g) {
    static_assert(KS == 1 || KS == 4, "slice_sync names four barriers");
    constexpr int NT = (TM / MR) * (TN / 4), LA = TM * GK / NT, LB = TN * GK / NT;
    __shared__ __align__(16) float As[KS][GK][TM + 4], Bs[KS][GK][TN + 4];
    static_assert(KS == 1 || KS * TM * TN <= KS * GK * (TM + 4), "the slice sums are staged in As");
    const int tid = threadIdx.x % NT, slice = threadIdx.x / NT, tx = tid % (TN / 4), ty = tid / (TN / 4), z = blockIdx.z;
    const int i0 = blockIdx.x * TM, j0 = blockIdx.y * TN;
    auto slice_sync = [&]() {
        if (KS == 1) __syncthreads();
        else if (slice == 0) asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");   // literal ids: ptxas reserves all 16 otherwise
        else if (slice == 1) asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory");
        else if (slice == 2) asm volatile("bar.sync 3, %0;" ::"n"(NT) : "memory");
        else asm volatile("bar.sync 4, %0;" ::"n"(NT) : "memory");
    };
    float acc[MR][4];
#pragma unroll
    for (int a = 0; a < MR; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = 0.f;
    float ra[LA], rb[LB];
    // A thread's elements of a chunk share ONE feature index and step through rows with a constant stride, so a chunk
    // costs one address computation per operand; the loads are unconditional (a safe address when out of range) and
    // therefore all in flight together.  RS = row step between a thread's consecutive elements.
    constexpr int RSA = AO ? NT / GK : NT / TM, RSB = BO ? NT / GK : NT / TN;
    static_assert(NT % GK == 0 && NT % TM == 0 && NT % TN == 0, "thread count must tile the chunk");
    const int fa_off = AO ? tid % GK : tid % TM, ra_off = AO ? tid / GK : tid / TM;
    const int fb_off = BO ? tid % GK : tid % TN, rb_off = BO ? tid / GK : tid / TN;
    auto fetch_one = [&](const Mat &m, bool out_is_row, int out0, int out_lim, int c0, int f_off, int r_off, int rs, float *dst, int n) {
        const int f = (out_is_row ? c0 : out0) + f_off, row0 = (out_is_row ? out0 : c0) + r_off;
        const int f_lim = out_is_row ? g.Kc : out_lim, row_lim = out_is_row ? out_lim : g.Kc;
        const bool second = f >= m.split;
        const float *base = second ? m.p2 + z * m.net_stride2 + (f - m.split) : m.p1 + z * m.net_stride1 + f;
        const int ld = second ? m.ld2 : m.ld1;
        const bool f_ok = f < f_lim && f != m.ones_at;
        const float *p = base + (size_t)row0 * ld;
        const size_t step = (size_t)rs * ld;
#pragma unroll
        for (int u = 0; u < n; u++) {
            dst[u] = __ldg((f_ok && row0 + u * rs < row_lim) ? p : m.p1);
            p += step;
        }
    };
    auto fetch = [&](int c0) {
        fetch_one(g.A, AO, i0, g.Mo, c0, fa_off, ra_off, RSA, ra, LA);
        fetch_one(g.B, BO, j0, g.No, c0, fb_off, rb_off, RSB, rb, LB);
    };
    if (slice * GK < g.Kc) fetch(slice * GK);
    for (int c0 = slice * GK; c0 < g.Kc; c0 += KS * GK) {
        {
            const int f = (AO ? c0 : i0) + fa_off, f_lim = AO ? g.Kc : g.Mo, row_lim = AO ? g.Mo : g.Kc, row0 = (AO ? i0 : c0) + ra_off;
            const bool one = f == g.A.ones_at && f < f_lim, f_ok = f < f_lim;
#pragma unroll
            for (int u = 0; u < LA; u++) {
                const float v = (f_ok && row0 + u * RSA < row_lim) ? (one ? 1.f : ra[u]) : 0.f;
                if (AO) As[slice][fa_off][ra_off + u * RSA] = v; else As[slice][ra_off + u * RSA][fa_off] = v;
            }
        }
        {
            const int f = (BO ? c0 : j0) + fb_off, f_lim = BO ? g.Kc : g.No, row_lim = BO ? g.No : g.Kc, row0 = (BO ? j0 : c0) + rb_off;
            const bool one = f == g.B.ones_at && f < f_lim, f_ok = f < f_lim;
#pragma unroll
            for (int u = 0; u < LB; u++) {
                const float v = (f_ok && row0 + u * RSB < row_lim) ? (one ? 1.f : rb[u]) : 0.f;
                if (BO) Bs[slice][fb_off][rb_off + u * RSB] = v; else Bs[slice][rb_off + u * RSB][fb_off] = v;
            }
        }
        slice_sync();
        if (c0 + KS * GK < g.Kc) fetch(c0 + KS * GK);
#pragma unroll
        for (int c = 0; c < GK; c++) {
            float av[MR];
            if constexpr (MR == 4) {
                const float4 a = *reinterpret_cast<const float4 *>(&As[slice][c][ty * 4]);
                av[0] = a.x; av[1] = a.y; av[2] = a.z; av[3] = a.w;
            } else {
                const float2 a = *reinterpret_cast<const float2 *>(&As[slice][c][ty * 2]);
                av[0] = a.x; av[1] = a.y;
            }
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[slice][c][tx * 4]);
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int p = 0; p < MR; p++)
#pragma unroll
                for (int q = 0; q < 4; q++) acc[p][q] = fmaf(av[p], bv[q], acc[p][q]);
        }
        slice_sync();
    }
    if constexpr (KS == 1) {
#pragma unroll
        for (int p = 0; p < MR; p++) {
            const int i = i0 + ty * MR + p;
            if (i >= g.Mo) continue;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int j = j0 + tx * 4 + q;
                if (j < g.No) gemm_emit(g, z, i, j, acc[p][q]);
            }
        }
    } else {
        __syncthreads();                                           // every slice is done with As / Bs
        float *red = &As[0][0][0];                                 // [KS][TM][TN]
#pragma unroll
        for (int p = 0; p < MR; p++)
            *reinterpret_cast<float4 *>(red + ((size_t)slice * TM + ty * MR + p) * TN + tx * 4) = make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]);
        __syncthreads();
        for (int o = threadIdx.x; o < TM * TN; o += NT * KS) {    // coalesced along j; slices added in the order 0, 1, ...
            float v = red[o];
#pragma unroll
            for (int s2 = 1; s2 < KS; s2++) v += red[(size_t)s2 * TM * TN + o];
            const int i = i0 + o / TN, j = j0 + o % TN;
            if (i < g.Mo && j < g.No) gemm_emit(g, z, i, j, v);
        }
    }
}

// gemm_tc.cu: the same contraction on tcgen05 (3xTF32).  Returns false when the engine is off / the shape is not covered.
bool gemm_tc_launch(const GemmArgs &g, int nets, bool ao, bool bo, cudaStream_t st, int engine);
// the TS form (the 128-row operand in tensor memory); gs in the kernel's own orientation, see gemm_tc.cu
bool gemm_ts_launch(const GemmArgs &gs, int nets, bool bo, bool swap, cudaStream_t st, int engine);
void transpose_weights(int rows, int cols, int nets, const float *src, float *dst, cudaStream_t st);
cudaError_t gemm_tc_prepare();

struct GemmLauncher {
    cudaStream_t st;
    int count = 0;
    long long *stamps = nullptr;
    bool fixed_order = false;   // SIMT tiles: never slice the contraction axis (a row's sum must not depend on the launch's shape)
    int engine = -1;   // -1: library default (prl_set_contraction_engine); 0: SIMT tiles; 1 / 64 / 32: tcgen05 tiles
    template <bool AO, bool BO>
    void run(const GemmArgs &g, int nets) {
        if (stamps) { GemmArgs gs = g; gs.stamps = stamps; if (gemm_tc_launch(gs, nets, AO, BO, st, engine)) { count++; return; } }
        if (gemm_tc_launch(g, nets, AO, BO, st, engine)) { count++; return; }
        const long long big = (long long)((g.Mo + 63) / 64) * ((g.No + 63) / 64) * nets;
        if (big >= 96) {       // enough 64x64 tiles to occupy the chip
            dim3 grid((g.Mo + 63) / 64, (g.No + 63) / 64, nets);
            k_gemm<64, 64, 4, 1, AO, BO><<<grid, 256, 0, st>>>(g);
        } else {               // small problem: 4x the CTAs, 4 warps each (2 x 4 outputs per thread), x 4 K slices
            dim3 grid((g.Mo + 31) / 32, (g.No + 31) / 32, nets);
            if (g.Kc > 2 * GK && !fixed_order) k_gemm<32, 32, 2, 4, AO, BO><<<grid, 512, 0, st>>>(g);
            else k_gemm<32, 32, 2, 1, AO, BO><<<grid, 128, 0, st>>>(g);
        }
        count++;
    }
    static GemmArgs base() {
        GemmArgs g;
        memset(&g, 0, sizeof(g));
        g.tail_col = -1;
        return g;
    }
    // y[M x N] = act(x W^T + b).  Wt (optional): W transposed, [K x N] with row pitch ldwt — offered to the TS-form kernel
    void fwd(Mat X, int M, const float *W, int ldw, long long w_ns, const float *b, long long b_ns, int N, int K, bool relu, float *Y,
             int ldy, long long y_ns, int nets = 1, const float *Wt = nullptr, int ldwt = 0, long long wt_ns = 0) {
        GemmArgs g = base();
        g.Mo = M; g.No = N; g.Kc = K; g.C = Y; g.ldc = ldy; g.c_net_stride = y_ns; g.bias = b; g.bias_net_stride = b_ns; g.relu = relu;
        if (Wt) {                                        // D[n][m] = sum_k Wt[k][n] x[m][k]
            GemmArgs t = g;
            t.A = mat(Wt, ldwt, wt_ns); t.B = X; t.Mo = N; t.No = M; t.stamps = stamps;
            if (gemm_ts_launch(t, nets, true, true, st, engine)) { count++; return; }
        }
        g.A = X; g.B = mat(W, ldw, w_ns);
        run<true, true>(g, nets);
    }
    // dx[M x Kx] (+)= dy[M x N] W[:, col0 : col0 + Kx]   (kept only where mask > 0)
    void bwd_x(const float *dY, int ldy, long long dy_ns, int M, int N, const float *W, int ldw, long long w_ns, int col0, int Kx, float *dX,
               int ldx, long long dx_ns, const float *mask, int ldm, long long m_ns, bool accumulate, int nets = 1) {
        GemmArgs g = base();
        g.A = mat(dY, ldy, dy_ns);
        g.B = mat(W + col0, ldw, w_ns);                  // B(out = k, c = n) = W[n][col0 + k]
        g.Mo = M; g.No = Kx; g.Kc = N; g.C = dX; g.ldc = ldx; g.c_net_stride = dx_ns;
        g.mask = mask; g.ldm = ldm; g.mask_net_stride = m_ns; g.accumulate = accumulate;
        {                                                // D[k][m] = sum_n W[n][col0 + k] dy[m][n]
            GemmArgs t = g;
            t.A = g.B; t.B = g.A; t.Mo = Kx; t.No = M; t.stamps = stamps;
            if (gemm_ts_launch(t, nets, true, true, st, engine)) { count++; return; }
        }
        run<true, false>(g, nets);
    }
    // dW[N x K] = dy^T x ; db[N] = column sums of dy (x extended with a ones column)
    void bwd_w(const float *dY, int ldy, long long dy_ns, int M, int N, Mat X, int K, float *dW, int ldw, long long dw_ns, float *db,
               long long db_ns, int nets = 1) {
        GemmArgs g = base();
        g.A = mat(dY, ldy, dy_ns);                       // A(out = n, c = m) = dy[m][n]
        X.ones_at = K;
        g.B = X;                                         // B(out = k, c = m) = x[m][k]
        g.Mo = N; g.No = K + 1; g.Kc = M; g.C = dW; g.ldc = ldw; g.c_net_stride = dw_ns;
        g.C_tail = db; g.tail_col = K; g.tail_net_stride = db_ns;
        {
            GemmArgs t = g;
            t.stamps = stamps;
            if (gemm_ts_launch(t, nets, false, false, st, engine)) { count++; return; }
        }
        run<false, false>(g, nets);
    }
};

// ------------------------------------------------------------------ pieces shared by the actor-critic learners
// dC2[z][m][j] = dq[z][m] * W3[z][j] * (c2 > 0)      (backward through the scalar head)
static __global__ void k_head_bwd(int B, int H, const float *__restrict__ dq, const float *__restrict__ w3, long long w_net_stride,
                           const float *__restrict__ c2, float *__restrict__ dc2) {
    const int z = blockIdx.z;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * H) return;
    const int m = e / H, j = e - m * H;
    const size_t o = (size_t)z * B * H + e;
    dc2[o] = (c2[o] > 0.f) ? dq[z * B + m] * __ldg(w3 + z * w_net_stride + j) : 0.f;
}

// twin-critic MSE (critic_utils.py:170-203): loss = (mse(q1, y) + mse(q2, y)) / 2 with q = [2][B], and its gradient
// dq_i = (q_i - y) / B.  Called by every thread of ONE block of 256 (fixed summation order); the loss is returned to thread 0.
__device__ __forceinline__ float twin_mse_block(int B, const float *__restrict__ q, const float *__restrict__ y, float *__restrict__ dq) {
    __shared__ float red[256];
    float s = 0.f;
    const float ib = 1.f / (float)B;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const float e1 = q[b] - y[b], e2 = q[B + b] - y[b];
        s += e1 * e1 + e2 * e2;
        dq[b] = e1 * ib;            // d/dq1 of (mse1 + mse2) / 2
        dq[B + b] = e2 * ib;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    return red[0] * ib * 0.5f;
}

struct AdamHp { float decay, omb1, beta2, omb2, eps; };
__device__ __forceinline__ float adamw1(float w, float &m, float &v, float &x, float g, const AdamHp &h, float step_size, float bc2s) {
    float p = __fmul_rn(w, h.decay);
    m = fmaf(h.omb1, g - m, m);
    v = __fadd_rn(__fmul_rn(v, h.beta2), __fmul_rn(__fmul_rn(h.omb2, g), g));
    x = fmaxf(x, v);
    const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(x), bc2s), h.eps);
    return __fadd_rn(p, __fdiv_rn(__fmul_rn(-step_size, m), denom));
}
// AdamW(amsgrad) over a flat vector; optional soft update of a target vector with the NEW parameters
static __global__ void k_adamw(int n, float *__restrict__ w, float *__restrict__ m, float *__restrict__ v, float *__restrict__ vmax,
                        const float *__restrict__ grad, AdamHp h, const float2 *__restrict__ scal, const int *__restrict__ round_idx,
                        float *__restrict__ target, float tau, float omtau) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 sc = scal[*round_idx];
    float mm = m[i], vv = v[i], xx = vmax[i];
    const float p = adamw1(w[i], mm, vv, xx, grad[i], h, sc.x, sc.y);
    w[i] = p; m[i] = mm; v[i] = vv; vmax[i] = xx;
    if (target) target[i] = __fadd_rn(__fmul_rn(tau, p), __fmul_rn(omtau, target[i]));
}
inline AdamHp adam_hp(double lr, double beta1, double beta2, double eps, double weight_decay) {
    return AdamHp{(float)(1.0 - lr * weight_decay), (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)eps};
}

}  // namespace prl
