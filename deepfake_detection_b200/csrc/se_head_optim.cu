// Small per-image kernels (squeeze-excite FCs, classifier + cross-entropy loss) and the flat-arena
// optimizer / weight-preparation kernels.
//
// Reference semantics restated here:
//   SqueezeExcite.forward         dfd/timm/models/efficientnet_blocks.py:104-110  (FC+bias, Swish, FC+bias, sigmoid)
//   classifier + loss             dfd/timm/models/efficientnet.py:348, dfd/timm/loss/cross_entropy.py:20-36,
//                                 nn.CrossEntropyLoss (dfd/runners/train.py:509-520); 2-class CE == sigmoid-BCE on z1-z0,
//                                 any other class count: softmax-CE (head_loss_kernel)
//   accuracy                      dfd/timm/utils.py:170-186
//   SGD nesterov                  torch.optim.SGD as configured by dfd/timm/optim/optim_factory.py:48-50
//   Adam / AdamW                  optim_factory.py:51-56, dfd/timm/optim/adamw.py:55-117
//   RMSpropTF                     dfd/timm/optim/rmsprop_tf.py:57-122
#include "common.cuh"

namespace {

// Scratch of the small batch-reduction kernels below (SE / classifier parameter gradients, the loss): split partial sums
// land in fixed slots and the last CTA of a group to arrive (ticket) adds them in slot order, so the results do not depend
// on CTA arrival order. Library-owned (zero at load, tickets self-reset); the kernels of one process run on one stream.
constexpr int SMALL_WS_FLOATS = 1 << 20;
constexpr int SMALL_TICKETS = 8192;
__device__ float g_small_ws[SMALL_WS_FLOATS];
__device__ int g_small_tk[SMALL_TICKETS];

__device__ __forceinline__ bool ticket_last(int* counter, int total) {
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const int t = atomicAdd(counter, 1);
        s_last = (t == total - 1);
        if (s_last) *counter = 0;
    }
    __syncthreads();
    const bool last = s_last != 0;
    if (last) __threadfence();
    return last;
}

__device__ __forceinline__ float swish_precise(float x) { return x * sigmoid_precise(x); }
__device__ __forceinline__ float softplus_precise(float x) {
    // log(1 + exp(x)), stable
    return fmaxf(x, 0.f) + log1pf(__expf(-fabsf(x)));
}

// ---------------------------------------------------------------------------------------------
// SE excite: gate[n,:] = sigmoid(We * swish(Wr * pooled[n,:] + br) + be).  A CTA handles IMG images: every weight element
// is fetched once per CTA and used for IMG images (with one image per CTA the 256 CTAs of a batch re-read both weight
// matrices - 113 MB of L2 traffic for the 1152-channel layers, which is what bounded this kernel at ~20 us).  The arithmetic
// order per image does not depend on IMG.
// ---------------------------------------------------------------------------------------------
template <int IMG>
__global__ void se_fc_fwd_kernel(const float* __restrict__ pooled, const float* __restrict__ Wr,
                                 const float* __restrict__ br, const float* __restrict__ We,
                                 const float* __restrict__ be, float* __restrict__ gate, int N, int C, int Cse) {
    extern __shared__ float sm[];
    float* p = sm;                 // [IMG][C]
    float* r = sm + IMG * C;       // [IMG][Cse]
    const int n0 = blockIdx.x * IMG, tid = threadIdx.x, nt = blockDim.x;
    const int ni = min(IMG, N - n0);
    for (int e = tid; e < IMG * C; e += nt) {
        const int i = e / C;
        p[e] = i < ni ? pooled[(size_t)n0 * C + e] : 0.f;
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
    for (int j = warp; j < Cse; j += nw) {
        const float* w = Wr + (size_t)j * C;
        float s[IMG];
#pragma unroll
        for (int i = 0; i < IMG; i++) s[i] = 0.f;
        for (int c = lane; c < C; c += 32) {
            const float wv = w[c];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, p[i * C + c], s[i]);
        }
        const float bj = br[j];
#pragma unroll
        for (int i = 0; i < IMG; i++) {
            const float t = warp_sum(s[i]);
            if (lane == 0) r[i * Cse + j] = swish_precise(t + bj);
        }
    }
    __syncthreads();
    // one thread per output row: a row is Cse consecutive floats, so the warp's 32 rows stay L1-resident across the j loop
    for (int c = tid; c < C; c += nt) {
        const float* w = We + (size_t)c * Cse;
        float s[IMG];
        const float bc = be[c];
#pragma unroll
        for (int i = 0; i < IMG; i++) s[i] = bc;
        for (int j = 0; j < Cse; j++) {
            const float wv = w[j];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, r[i * Cse + j], s[i]);
        }
#pragma unroll
        for (int i = 0; i < IMG; i++)
            if (i < ni) gate[(size_t)(n0 + i) * C + c] = sigmoid_precise(s[i]);
    }
}

// SE backward, IMG images per CTA: from draw = dL/dgate recompute the FC chain and emit
//   d_e [N,C], r [N,Cse], d_rpre [N,Cse] (for the parameter-gradient kernel) and dpool [N,C].
template <int IMG>
__global__ void se_fc_bwd_kernel(const float* __restrict__ draw, const float* __restrict__ pooled,
                                 const float* __restrict__ Wr, const float* __restrict__ br,
                                 const float* __restrict__ We, const float* __restrict__ be,
                                 float* __restrict__ d_e, float* __restrict__ r_out, float* __restrict__ d_rpre,
                                 float* __restrict__ dpool, int N, int C, int Cse) {
    extern __shared__ float sm[];
    float* p = sm;                         // [IMG][C]
    float* de = p + IMG * C;               // [IMG][C]
    float* rpre = de + IMG * C;            // [IMG][Cse]
    float* r = rpre + IMG * Cse;           // [IMG][Cse]
    float* drp = r + IMG * Cse;            // [IMG][Cse]
    float* r_part = drp + IMG * Cse;       // [warps][IMG][Cse] per-warp partials of d_r, summed in warp order
    const int n0 = blockIdx.x * IMG, tid = threadIdx.x, nt = blockDim.x;
    const int ni = min(IMG, N - n0);
    for (int e = tid; e < IMG * C; e += nt) {
        const int i = e / C;
        p[e] = i < ni ? pooled[(size_t)n0 * C + e] : 0.f;
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
    for (int j = warp; j < Cse; j += nw) {
        const float* w = Wr + (size_t)j * C;
        float s[IMG];
#pragma unroll
        for (int i = 0; i < IMG; i++) s[i] = 0.f;
        for (int c = lane; c < C; c += 32) {
            const float wv = w[c];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, p[i * C + c], s[i]);
        }
        const float bj = br[j];
#pragma unroll
        for (int i = 0; i < IMG; i++) {
            const float t = warp_sum(s[i]);
            if (lane == 0) { rpre[i * Cse + j] = t + bj; r[i * Cse + j] = swish_precise(t + bj); }
        }
    }
    __syncthreads();
    for (int c = tid; c < C; c += nt) {
        const float* w = We + (size_t)c * Cse;
        float s[IMG];
        const float bc = be[c];
#pragma unroll
        for (int i = 0; i < IMG; i++) s[i] = bc;
        for (int j = 0; j < Cse; j++) {
            const float wv = w[j];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, r[i * Cse + j], s[i]);
        }
#pragma unroll
        for (int i = 0; i < IMG; i++) {
            float v = 0.f;
            if (i < ni) {
                const float g = sigmoid_precise(s[i]);
                v = draw[(size_t)(n0 + i) * C + c] * g * (1.f - g);
                d_e[(size_t)(n0 + i) * C + c] = v;
            }
            de[i * C + c] = v;
        }
    }
    __syncthreads();
    // d_r[i][j] = sum_c We[c,j] * de[i][c]: lanes walk j (contiguous in We's rows), warps split c; partials meet in smem
    for (int j0 = 0; j0 < Cse; j0 += 32) {
        const int j = j0 + lane;
        if (j < Cse) {
            float s[IMG];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = 0.f;
            for (int c = warp; c < C; c += nw) {
                const float wv = We[(size_t)c * Cse + j];
#pragma unroll
                for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, de[i * C + c], s[i]);
            }
#pragma unroll
            for (int i = 0; i < IMG; i++) r_part[(warp * IMG + i) * Cse + j] = s[i];
        }
    }
    __syncthreads();
    for (int e = tid; e < IMG * Cse; e += nt) {
        const int i = e / Cse, j = e - i * Cse;
        float s = 0.f;
        for (int w = 0; w < nw; w++) s += r_part[(w * IMG + i) * Cse + j];
        const float x = rpre[e];
        const float sg = sigmoid_precise(x);
        const float v = s * (sg * (1.f + x * (1.f - sg)));
        drp[e] = v;
        if (i < ni) {
            d_rpre[(size_t)(n0 + i) * Cse + j] = v;
            r_out[(size_t)(n0 + i) * Cse + j] = r[e];
        }
    }
    __syncthreads();
    for (int c = tid; c < C; c += nt) {
        float s[IMG];
#pragma unroll
        for (int i = 0; i < IMG; i++) s[i] = 0.f;
        for (int j = 0; j < Cse; j++) {
            const float wv = Wr[(size_t)j * C + c];
#pragma unroll
            for (int i = 0; i < IMG; i++) s[i] = fmaf(wv, drp[i * Cse + j], s[i]);
        }
#pragma unroll
        for (int i = 0; i < IMG; i++)
            if (i < ni) dpool[(size_t)(n0 + i) * C + c] = s[i];
    }
}

// SE parameter gradients: one thread per (c, j); contraction over the N images.
__global__ void se_fc_wgrad_kernel(const float* __restrict__ d_e, const float* __restrict__ r,
                                   const float* __restrict__ d_rpre, const float* __restrict__ pooled,
                                   float* __restrict__ dWr, float* __restrict__ dbr, float* __restrict__ dWe,
                                   float* __restrict__ dbe, int N, int C, int Cse) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < C * Cse;
    const int c = valid ? idx / Cse : 0, j = valid ? idx - c * Cse : 0;
    // blockIdx.y splits the images so that the serial chain per thread stays short; the split partials go to fixed slots
    // [split][block][4][128] and are added in split order by the last block of this column group (ticket)
    const int per = (N + gridDim.y - 1) / gridDim.y;
    const int n0 = blockIdx.y * per, n1 = min(N, n0 + per);
    float awe = 0.f, awr = 0.f, abe = 0.f, abr = 0.f;
    if (valid) {
#pragma unroll 4
        for (int n = n0; n < n1; n++) {
            float de = d_e[(size_t)n * C + c], rr = r[(size_t)n * Cse + j];
            float dr = d_rpre[(size_t)n * Cse + j], pp = pooled[(size_t)n * C + c];
            awe = fmaf(de, rr, awe);
            awr = fmaf(dr, pp, awr);
            abe += de;
            abr += dr;
        }
    }
    if (gridDim.y > 1) {
        float* slot = g_small_ws + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 512;
        slot[threadIdx.x] = awe; slot[128 + threadIdx.x] = awr; slot[256 + threadIdx.x] = abe; slot[384 + threadIdx.x] = abr;
        if (!ticket_last(g_small_tk + blockIdx.x, gridDim.y)) return;
        awe = awr = abe = abr = 0.f;
        for (int y = 0; y < (int)gridDim.y; y++) {
            const float* sl = g_small_ws + ((size_t)y * gridDim.x + blockIdx.x) * 512;
            awe += __ldcg(sl + threadIdx.x); awr += __ldcg(sl + 128 + threadIdx.x);
            abe += __ldcg(sl + 256 + threadIdx.x); abr += __ldcg(sl + 384 + threadIdx.x);
        }
    }
    if (!valid) return;
    dWe[(size_t)c * Cse + j] += awe;
    dWr[(size_t)j * C + c] += awr;
    if (j == 0) dbe[c] += abe;
    if (c == 0) dbr[j] += abr;
}

// ---------------------------------------------------------------------------------------------
// 2-class classifier: logits[n,k] = W[k,:] . pooled[n,:] + b[k]   (one CTA per image, one warp per class round-robin)
// fused 2-class loss (sigmoid-BCE on d = z1 - z0 == softmax-CE), top-1, and dL/dlogits.
// target: int64 hard labels (tgt_i) or float soft targets [N,2] (tgt_f).
// ---------------------------------------------------------------------------------------------
__global__ void head_fwd_kernel(const float* __restrict__ pooled, const float* __restrict__ W,
                                const float* __restrict__ b, float* __restrict__ logits, int F, int K,
                                const long long* __restrict__ tgt_i, const float* __restrict__ tgt_f, float smoothing,
                                float inv_n, float loss_scale, const float* __restrict__ loss_scale_dev,
                                float* __restrict__ loss_acc, float* __restrict__ correct_acc,
                                float* __restrict__ dlogits) {
    __shared__ float z[32];
    const int n = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const float* p = pooled + (size_t)n * F;
    for (int k = warp; k < K; k += nw) {
        const float* w = W + (size_t)k * F;
        float s = 0.f;
        for (int f = lane; f < F; f += 32) s = fmaf(w[f], p[f], s);
        s = warp_sum(s);
        if (lane == 0) { z[k] = s + b[k]; logits[(size_t)n * K + k] = s + b[k]; }
    }
    if (!loss_acc) return;
    __syncthreads();
    if (threadIdx.x == 0 && K == 2) {
        float t0, t1;
        if (tgt_f) { t0 = tgt_f[n * 2]; t1 = tgt_f[n * 2 + 1]; }
        else {
            int y = (int)tgt_i[n];
            t1 = y ? 1.f - 0.5f * smoothing : 0.5f * smoothing;
            t0 = y ? 0.5f * smoothing : 1.f - 0.5f * smoothing;
        }
        float d = z[1] - z[0];
        float loss = t0 * softplus_precise(d) + t1 * softplus_precise(-d);
        float sg = sigmoid_precise(d);
        float g1 = (t0 + t1) * sg - t1;
        int pred = z[1] > z[0] ? 1 : 0;      // topk(1) returns the first index on ties
        int lab = t1 > t0 ? 1 : 0;
        // per-image loss / hit in fixed slots; the last image's CTA adds them in image order (below)
        g_small_ws[n] = loss * inv_n;
        g_small_ws[gridDim.x + n] = pred == lab ? 1.f : 0.f;
        if (dlogits) {
            const float ls = loss_scale_dev ? loss_scale * *loss_scale_dev : loss_scale;   // fp16 dynamic loss scaling
            dlogits[n * 2] = -g1 * inv_n * ls;
            dlogits[n * 2 + 1] = g1 * inv_n * ls;
        }
    }
    if (K != 2) return;
    if (!ticket_last(g_small_tk, gridDim.x)) return;
    if (threadIdx.x == 0) {
        float l = 0.f, c = 0.f;
        for (int i = 0; i < (int)gridDim.x; i++) { l += __ldcg(g_small_ws + i); c += __ldcg(g_small_ws + gridDim.x + i); }
        *loss_acc += l;
        *correct_acc += c;
    }
}

// dpooled[n,f] = sum_k dlogits[n,k] W[k,f]
__global__ void head_dgrad_kernel(const float* __restrict__ dlogits, const float* __restrict__ W,
                                  float* __restrict__ dpooled, int N, int F, int K) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)N * F) return;
    int n = (int)(idx / F), f = (int)(idx - (size_t)n * F);
    float s = 0.f;
    for (int k = 0; k < K; k++) s = fmaf(dlogits[(size_t)n * K + k], W[(size_t)k * F + f], s);
    dpooled[idx] = s;
}
// dW[k,f] += sum_n dlogits[n,k] pooled[n,f]; db[k] += sum_n dlogits[n,k]; the batch is split over blockIdx.y
// (a single thread walking all N images serialises N dependent L2 round trips: measured 100 us at N = 256)
__global__ void head_wgrad_kernel(const float* __restrict__ dlogits, const float* __restrict__ pooled,
                                  float* __restrict__ dW, float* __restrict__ db, int N, int F, int K) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < K * F;
    const int k = valid ? idx / F : 0, f = valid ? idx - k * F : 0;
    const int per = (N + gridDim.y - 1) / gridDim.y;
    const int n0 = blockIdx.y * per, n1 = min(N, n0 + per);
    float s = 0.f, sb = 0.f;
    if (valid) {
#pragma unroll 4
        for (int n = n0; n < n1; n++) {
            float d = dlogits[(size_t)n * K + k];
            s = fmaf(d, pooled[(size_t)n * F + f], s);
            sb += d;
        }
    }
    // fixed-slot split partials, added in split order by the last block of the column group (no atomics)
    float* slot = g_small_ws + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 256;
    slot[threadIdx.x] = s; slot[128 + threadIdx.x] = sb;
    if (!ticket_last(g_small_tk + blockIdx.x, gridDim.y)) return;
    if (!valid) return;
    s = sb = 0.f;
    for (int y = 0; y < (int)gridDim.y; y++) {
        const float* sl = g_small_ws + ((size_t)y * gridDim.x + blockIdx.x) * 256;
        s += __ldcg(sl + threadIdx.x); sb += __ldcg(sl + 128 + threadIdx.x);
    }
    dW[idx] += s;
    if (f == 0) db[k] += sb;
}

// ---------------------------------------------------------------------------------------------
// K-class head (every K != 2 up to HEAD_KMAX): softmax cross-entropy with the reference's three target encodings.
// The three products of the classifier run through one fp32 tile kernel; the loss / top-1 / dL/dlogits run one CTA per
// image row.  Every output is a single fixed-order sum (no split partials, no atomics), so results are bit-reproducible.
// ---------------------------------------------------------------------------------------------
constexpr int HEAD_KMAX = 4096;
constexpr int HG_BK = 16;            // contraction depth of one shared-memory stage
constexpr int HL_THREADS = 256;

// C[m, c] (+)= sum_r A(m, r) B(r, c) (+ bias[c]).  A(m, r) = A[m*lda + r] if A_RC (contraction index contiguous), else
// A[r*lda + m]; B(r, c) = B[c*ldb + r] if B_RC, else B[r*ldb + c].  A BM x BN tile per CTA, 4 x 4 outputs per thread; the
// next HG_BK-deep stage is loaded into registers while the current one is multiplied out of shared memory.  Every output
// accumulates r = 0, 1, ..., R-1 in order whatever the tile shape, so the launcher's tile choice never changes a bit.
template <int BM, int BN, bool A_RC, bool B_RC>
__global__ void __launch_bounds__((BM / 4) * (BN / 4))
head_gemm_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                 const float* __restrict__ bias, int accumulate, int M, int Nc, int R) {
    constexpr int NT = (BM / 4) * (BN / 4), LA = HG_BK * BM / NT, LB = HG_BK * BN / NT;
    __shared__ __align__(16) float As[HG_BK][BM + 4];
    __shared__ __align__(16) float Bs[HG_BK][BN + 4];
    const int tid = threadIdx.x, tx = tid % (BN / 4), ty = tid / (BN / 4);
    const int m0 = blockIdx.y * BM, c0 = blockIdx.x * BN;
    float ra[LA], rb[LB];
    // element e of a stage: the operand's contiguous index runs fastest across the threads (coalesced loads)
    auto fetch = [&](int r0) {
#pragma unroll
        for (int i = 0; i < LA; i++) {
            const int e = tid + i * NT;
            const int r = A_RC ? e % HG_BK : e / BM, m = A_RC ? e / HG_BK : e % BM;
            const int gm = m0 + m, gr = r0 + r;
            ra[i] = (gm < M && gr < R) ? (A_RC ? A[(size_t)gm * lda + gr] : A[(size_t)gr * lda + gm]) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < LB; i++) {
            const int e = tid + i * NT;
            const int r = B_RC ? e % HG_BK : e / BN, c = B_RC ? e / HG_BK : e % BN;
            const int gc = c0 + c, gr = r0 + r;
            rb[i] = (gc < Nc && gr < R) ? (B_RC ? B[(size_t)gc * ldb + gr] : B[(size_t)gr * ldb + gc]) : 0.f;
        }
    };
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
    fetch(0);
    for (int r0 = 0; r0 < R; r0 += HG_BK) {
#pragma unroll
        for (int i = 0; i < LA; i++) {
            const int e = tid + i * NT;
            As[A_RC ? e % HG_BK : e / BM][A_RC ? e / HG_BK : e % BM] = ra[i];
        }
#pragma unroll
        for (int i = 0; i < LB; i++) {
            const int e = tid + i * NT;
            Bs[B_RC ? e % HG_BK : e / BN][B_RC ? e / HG_BK : e % BN] = rb[i];
        }
        __syncthreads();
        if (r0 + HG_BK < R) fetch(r0 + HG_BK);
#pragma unroll
        for (int r = 0; r < HG_BK; r++) {
            const float4 a = *reinterpret_cast<const float4*>(&As[r][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[r][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int c = c0 + tx * 4 + j;
            if (c >= Nc) continue;
            float* out = C + (size_t)m * ldc + c;
            float v = acc[i][j];
            if (bias) v += bias[c];
            *out = accumulate ? *out + v : v;
        }
    }
}

// block-wide sum in a fixed order (butterfly within warps, warp partials in warp order); every thread gets the result
__device__ __forceinline__ float block_sum_ordered(float v, float* red) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w];
    return s;
}

// block-wide (max, first index of the max); every thread gets the result
__device__ __forceinline__ void argmax_merge(float& v, int& i, float ov, int oi) {
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
}
__device__ __forceinline__ void block_argmax(float& v, int& i, float* redv, int* redi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) argmax_merge(v, i, __shfl_xor_sync(0xffffffffu, v, o), __shfl_xor_sync(0xffffffffu, i, o));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) { redv[warp] = v; redi[warp] = i; }
    __syncthreads();
    v = redv[0]; i = redi[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) argmax_merge(v, i, redv[w], redi[w]);
}

// one CTA per image row of logits [N, K]:
//   t_k = smoothing/K + (1 - smoothing)[k == y]  (hard label y, clamped into the row)  or  t = tgt_f[n, :] (soft),
//   loss_n = sum_k t_k (lse - z_k),  dlogits = (sum_k t_k * softmax(z) - t) / N * loss_scale,
//   pred = first index of the row max, label = y or the first argmax of the soft target row.
// The per-image loss / hit land in fixed slots and the last CTA adds them in image order (as head_fwd_kernel does).
__global__ void __launch_bounds__(HL_THREADS)
head_loss_kernel(const float* __restrict__ logits, int K, const long long* __restrict__ tgt_i,
                 const float* __restrict__ tgt_f, float smoothing, float inv_n, float loss_scale,
                 const float* __restrict__ loss_scale_dev, float* __restrict__ loss_acc, float* __restrict__ correct_acc,
                 float* __restrict__ dlogits) {
    __shared__ float redv[32];
    __shared__ int redi[32];
    const int n = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const float* z = logits + (size_t)n * K;
    const float* t = tgt_f ? tgt_f + (size_t)n * K : nullptr;
    float zmax = -INFINITY;
    int pred = K;
    for (int k = tid; k < K; k += nt) {
        const float v = z[k];
        if (pred == K || v > zmax) { zmax = v; pred = k; }
    }
    block_argmax(zmax, pred, redv, redi);
    int y = 0;
    if (!t) {
        const long long yl = tgt_i[n];
        y = yl < 0 ? 0 : (yl >= K ? K - 1 : (int)yl);
    }
    const float off = t ? 0.f : smoothing / (float)K, on = 1.f - smoothing + off;
    float se = 0.f, st = 0.f, tmax = -INFINITY;
    int lab = t ? K : y;
    for (int k = tid; k < K; k += nt) {
        se += expf(z[k] - zmax);
        if (t) {
            const float tk = t[k];
            st += tk;
            if (lab == K || tk > tmax) { tmax = tk; lab = k; }
        }
    }
    se = block_sum_ordered(se, redv);
    if (t) {
        st = block_sum_ordered(st, redv);
        block_argmax(tmax, lab, redv, redi);
    } else {
        st = 1.f;          // sum_k t_k is exactly 1 for a smoothed one-hot target
    }
    const float lse = zmax + logf(se);
    const float ls = (loss_scale_dev ? loss_scale * *loss_scale_dev : loss_scale) * inv_n;
    float loss = 0.f;
    for (int k = tid; k < K; k += nt) {
        const float v = z[k];
        const float tk = t ? t[k] : (k == y ? on : off);
        loss = fmaf(tk, lse - v, loss);
        if (dlogits) dlogits[(size_t)n * K + k] = (st * (expf(v - zmax) / se) - tk) * ls;
    }
    loss = block_sum_ordered(loss, redv);
    if (tid == 0) {
        g_small_ws[n] = loss * inv_n;
        g_small_ws[gridDim.x + n] = pred == lab ? 1.f : 0.f;
    }
    if (!ticket_last(g_small_tk, gridDim.x)) return;
    if (tid == 0) {
        float l = 0.f, c = 0.f;
        for (int i = 0; i < (int)gridDim.x; i++) { l += __ldcg(g_small_ws + i); c += __ldcg(g_small_ws + gridDim.x + i); }
        *loss_acc += l;
        *correct_acc += c;
    }
}

// db[k] += sum_n dlogits[n, k], images in order
__global__ void head_bias_grad_kernel(const float* __restrict__ dlogits, float* __restrict__ db, int N, int K) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    float s = 0.f;
#pragma unroll 8
    for (int n = 0; n < N; n++) s += dlogits[(size_t)n * K + k];
    db[k] += s;
}

// the tile shape: the largest of 64 x 64 / 32 x 64 / 32 x 32 that still gives the 148 SMs work (more, smaller CTAs for the
// small products of the head); results do not depend on it
template <bool A_RC, bool B_RC>
static int head_gemm(const float* A, int lda, const float* B, int ldb, float* C, int ldc, const float* bias, int accumulate,
                     int M, int Nc, int R, cudaStream_t st) {
    if ((long long)cdiv(M, 64) * cdiv(Nc, 64) >= 2 * 148)
        head_gemm_kernel<64, 64, A_RC, B_RC><<<dim3(cdiv(Nc, 64), cdiv(M, 64)), 256, 0, st>>>(A, lda, B, ldb, C, ldc, bias, accumulate, M, Nc, R);
    else if ((long long)cdiv(M, 32) * cdiv(Nc, 64) >= 148)
        head_gemm_kernel<32, 64, A_RC, B_RC><<<dim3(cdiv(Nc, 64), cdiv(M, 32)), 128, 0, st>>>(A, lda, B, ldb, C, ldc, bias, accumulate, M, Nc, R);
    else
        head_gemm_kernel<32, 32, A_RC, B_RC><<<dim3(cdiv(Nc, 32), cdiv(M, 32)), 64, 0, st>>>(A, lda, B, ldb, C, ldc, bias, accumulate, M, Nc, R);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

// ---------------------------------------------------------------------------------------------
// flat-arena optimizers.  One launch per parameter group (decay / no-decay ranges of the arena).
// g is multiplied by grad_scale (1/world for the DDP mean, 1/loss_scale for fp16) before use.
// If `skip` is non-null and *skip != 0 the step is skipped (fp16 overflow).  p16 (optional) receives the
// 16-bit copy of the updated weights that the GEMM / depthwise kernels read.
// ---------------------------------------------------------------------------------------------
template <typename T16>
__device__ __forceinline__ void store16(void* p16, size_t i, float v) {
    if (p16) reinterpret_cast<T16*>(p16)[i] = from_f<T16>(v);
}

template <typename T16>
__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, size_t n,
                           float lr, float momentum, float wd, int nesterov, float grad_scale,
                           const float* __restrict__ gscale_dev, const int* __restrict__ skip, void* __restrict__ p16,
                           const float* __restrict__ lr_dev) {
    if (skip && *skip) return;
    if (gscale_dev) grad_scale *= *gscale_dev;
    if (lr_dev) lr = *lr_dev;          // device-resident learning rate: one captured graph survives every scheduler update
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        float w = p[i];
        float gg = fmaf(wd, w, g[i] * grad_scale);
        float buf = fmaf(momentum, m[i], gg);     // first step: m == 0 -> buf = g (torch clones the gradient)
        m[i] = buf;
        float upd = nesterov ? fmaf(momentum, buf, gg) : buf;
        w = fmaf(-lr, upd, w);
        p[i] = w;
        store16<T16>(p16, i, w);
    }
}

template <typename T16>
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr, float b1, float b2, float eps, float wd,
                            int decoupled, float bc1, float bc2_sqrt, float grad_scale,
                            const float* __restrict__ gscale_dev, const int* __restrict__ skip, void* __restrict__ p16,
                            const float* __restrict__ lr_dev, const int* __restrict__ step_dev) {
    if (skip && *skip) return;
    if (gscale_dev) grad_scale *= *gscale_dev;
    if (lr_dev) lr = *lr_dev;
    if (step_dev) {                    // bias corrections from the device step counter (advanced by dfd_opt_tick)
        const float t = (float)*step_dev;
        bc1 = 1.f - powf(b1, t);
        bc2_sqrt = sqrtf(1.f - powf(b2, t));
    }
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        float w = p[i];
        float gg = g[i] * grad_scale;
        if (decoupled) w *= (1.f - lr * wd);       // adamw.py:72
        else gg = fmaf(wd, w, gg);                 // torch.optim.Adam L2
        float mm = fmaf(b1, m[i], (1.f - b1) * gg);
        float vv = fmaf(b2, v[i], (1.f - b2) * gg * gg);
        m[i] = mm;
        v[i] = vv;
        float denom = sqrtf(vv) / bc2_sqrt + eps;
        w -= (lr / bc1) * (mm / denom);
        p[i] = w;
        store16<T16>(p16, i, w);
    }
}

template <typename T16>
__global__ void rmsprop_tf_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ sq,
                                  float* __restrict__ mom, size_t n, float lr, float alpha, float eps, float wd,
                                  float momentum, float grad_scale, const float* __restrict__ gscale_dev,
                                  const int* __restrict__ skip, void* __restrict__ p16, const float* __restrict__ lr_dev) {
    if (skip && *skip) return;
    if (gscale_dev) grad_scale *= *gscale_dev;
    if (lr_dev) lr = *lr_dev;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        float w = p[i];
        float gg = fmaf(wd, w, g[i] * grad_scale);
        float s = sq[i];
        s = fmaf(1.f - alpha, gg * gg - s, s);     // rmsprop_tf.py:100 (TF op order)
        sq[i] = s;
        float avg = sqrtf(s + eps);                // eps inside the sqrt, :107
        if (momentum > 0.f) {
            float b = fmaf(momentum, mom[i], lr * gg / avg);   // lr folded into the buffer, :112-114
            mom[i] = b;
            w -= b;
        } else {
            w -= lr * gg / avg;
        }
        p[i] = w;
        store16<T16>(p16, i, w);
    }
}

// optimizer step counter on the device: advances unless the step is skipped (fp16 overflow), so Adam's bias correction
// follows apex semantics (a skipped step is not a step)
__global__ void opt_tick_kernel(int* __restrict__ step, const int* __restrict__ skip) {
    if (skip && *skip) return;
    *step += 1;
}

// up to 8 host scalars -> device floats (values travel as kernel arguments: nothing on the host has to stay alive)
struct F8 { float v[8]; };
__global__ void set_floats_kernel(float* __restrict__ dst, int n, F8 f) {
    if ((int)threadIdx.x < n) dst[threadIdx.x] = f.v[threadIdx.x];
}

// ModelEma.update (dfd/timm/utils.py:329-340) over a flat arena: ema = ema * decay + (1 - decay) * model
__global__ void ema_kernel(float* __restrict__ ema, const float* __restrict__ p, size_t n, float decay) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    const float om = 1.f - decay;
    for (; i < n; i += stride) ema[i] = ema[i] * decay + om * p[i];
}
// num_batches_tracked entries (int64): the reference computes in float and copy_() truncates back to int64
__global__ void ema_i64_kernel(long long* __restrict__ ema, const long long* __restrict__ p, int n, float decay) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ema[i] = (long long)((float)ema[i] * decay + (1.f - decay) * (float)p[i]);
}

template <typename T16>
__global__ void cast_arena_kernel(const float* __restrict__ p, T16* __restrict__ p16, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p16[i] = from_f<T16>(p[i]);
}

// any non-finite gradient -> *flag = 1   (fp16 dynamic loss scaling, apex O1 semantics train.py:353,632-634)
__global__ void check_finite_kernel(const float* __restrict__ g, size_t n, int* __restrict__ flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    int bad = 0;
    for (; i < n; i += stride) {
        float x = g[i];
        if (!(fabsf(x) <= 3.0e38f)) bad = 1;
    }
    if (bad) *flag = 1;
}

// dynamic loss scale update on the device (no host sync): halve on overflow, double after `interval` clean steps
__global__ void update_loss_scale_kernel(int* __restrict__ flag, float* __restrict__ scale, int* __restrict__ good,
                                         int interval, float* __restrict__ inv_scale_out) {
    if (*flag) {
        *scale = fmaxf(*scale * 0.5f, 1.f);
        *good = 0;
    } else {
        int g = *good + 1;
        if (g >= interval) { *scale = fminf(*scale * 2.f, 16777216.f); g = 0; }
        *good = g;
    }
    if (inv_scale_out) *inv_scale_out = 1.f / *scale;
    *flag = 0;        // consumed: the next step starts clean
}

// transposed 16-bit copies of the 1x1-conv weights for dgrad: src [O, I] -> dst [I, O]
struct TransposeDesc {
    const void* src;
    void* dst;
    int O;
    int I;
};
template <typename T16>
__global__ void transpose_weights_kernel(const TransposeDesc* __restrict__ table) {
    __shared__ T16 tile[32][33];
    TransposeDesc d = table[blockIdx.z];
    const T16* src = (const T16*)d.src;
    T16* dst = (T16*)d.dst;
    for (int o0 = blockIdx.y * 32; o0 < d.O; o0 += gridDim.y * 32) {
        for (int i0 = blockIdx.x * 32; i0 < d.I; i0 += gridDim.x * 32) {
            for (int r = threadIdx.y; r < 32; r += blockDim.y) {
                int o = o0 + r, i = i0 + threadIdx.x;
                if (o < d.O && i < d.I) tile[r][threadIdx.x] = src[(size_t)o * d.I + i];
            }
            __syncthreads();
            for (int r = threadIdx.y; r < 32; r += blockDim.y) {
                int i = i0 + r, o = o0 + threadIdx.x;
                if (o < d.O && i < d.I) dst[(size_t)i * d.O + o] = tile[threadIdx.x][r];
            }
            __syncthreads();
        }
    }
}

// The per-image FC chains are latency-bound (ncu: 8 % issue utilisation, long-scoreboard stalls, 0.2 waves): the only
// lever is a shorter dependent chain per warp, i.e. more warps per image for the wide layers.
static int se_threads(int C) { return C >= 768 ? 1024 : (C >= 384 ? 512 : 256); }

static int flat_blocks(size_t n) {
    size_t b = (n + 255) / 256;
    if (b > 148 * 8) b = 148 * 8;
    if (b < 1) b = 1;
    return (int)b;
}

// images per CTA of the SE FC kernels. Several images per CTA fetch every weight element once for all of them, but
// MEASURED (B0, batch 256): 4 images per CTA are 12 % slower than 1 (0.80 vs 0.69 ms over the 16 backward launches) - the
// kernels are bound by the dependent FC chain of a CTA, which gets longer, not by the L2 traffic of the weights. So: one
// image per CTA until the batch is so large that the grid exceeds a few waves - EXCEPT for the widest layers, where the
// weight traffic does bound the kernel (1152 x 48: 2 x 221 KB per CTA; per layer, weights L2-resident: forward 43 / 31 / 37 us
// and backward + wgrad 98 / 77 / 82 us for 1 / 2 / 4 images per CTA; 672 x 28 and below: 1 is best).
static int se_img(int N, int C, int Cse, size_t floats_per_image, size_t fixed_floats) {
    int img = N >= 2048 ? 4 : (N >= 1024 ? 2 : 1);
    if (img < 2 && N >= 128 && (long long)C * Cse >= 32768) img = 2;
    { static int f = -1; if (f < 0) { const char* e = getenv("DFD_SE_IMG"); f = e ? atoi(e) : 0; } if (f == 1 || f == 2 || f == 4) img = f; }
    while (img > 1 && (img * floats_per_image + fixed_floats) * sizeof(float) > 200 * 1024) img >>= 1;
    return img;
}

template <typename K>
static int se_smem_attr(K kern, size_t smem, bool* done) {
    if (smem > 48 * 1024 && !*done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return dfd_set_cuda_error(e, __FILE__, __LINE__);
        *done = true;
    }
    return smem > 200 * 1024 ? dfd_set_error(DFD_ERR_UNSUPPORTED, "squeeze-excite: channel count exceeds shared memory") : DFD_OK;
}

}  // namespace

extern "C" {

int dfd_se_fc_fwd(const float* pooled, const float* Wr, const float* br, const float* We, const float* be,
                  float* gate, int N, int C, int Cse, void* stream) {
    if (N <= 0 || C <= 0 || Cse <= 0) return dfd_set_error(DFD_ERR_ARG, "dfd_se_fc_fwd: sizes");
    const int img = se_img(N, C, Cse, (size_t)C + Cse, 0);
    const size_t smem = (size_t)img * (C + Cse) * sizeof(float);
    const int blocks = (N + img - 1) / img, nthr = se_threads(C);
    cudaStream_t st = (cudaStream_t)stream;
    static bool a4 = false, a2 = false, a1 = false;
    int rc;
    if (img == 4) { if ((rc = se_smem_attr(se_fc_fwd_kernel<4>, smem, &a4))) return rc; se_fc_fwd_kernel<4><<<blocks, nthr, smem, st>>>(pooled, Wr, br, We, be, gate, N, C, Cse); }
    else if (img == 2) { if ((rc = se_smem_attr(se_fc_fwd_kernel<2>, smem, &a2))) return rc; se_fc_fwd_kernel<2><<<blocks, nthr, smem, st>>>(pooled, Wr, br, We, be, gate, N, C, Cse); }
    else { if ((rc = se_smem_attr(se_fc_fwd_kernel<1>, smem, &a1))) return rc; se_fc_fwd_kernel<1><<<blocks, nthr, smem, st>>>(pooled, Wr, br, We, be, gate, N, C, Cse); }
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_se_fc_bwd(const float* draw, const float* pooled, const float* Wr, const float* br, const float* We,
                  const float* be, float* d_e, float* r, float* d_rpre, float* dpool, float* dWr, float* dbr,
                  float* dWe, float* dbe, int N, int C, int Cse, void* stream) {
    if (N <= 0 || C <= 0 || Cse <= 0) return dfd_set_error(DFD_ERR_ARG, "dfd_se_fc_bwd: sizes");
    const int nthr = se_threads(C), nw = nthr / 32;
    const int img = se_img(N, C, Cse, (size_t)2 * C + (size_t)(3 + nw) * Cse, 0);
    const size_t smem = (size_t)img * (2 * C + (3 + nw) * Cse) * sizeof(float);
    const int blocks = (N + img - 1) / img;
    cudaStream_t st = (cudaStream_t)stream;
    static bool a4 = false, a2 = false, a1 = false;
    int rc;
    if (img == 4) { if ((rc = se_smem_attr(se_fc_bwd_kernel<4>, smem, &a4))) return rc; se_fc_bwd_kernel<4><<<blocks, nthr, smem, st>>>(draw, pooled, Wr, br, We, be, d_e, r, d_rpre, dpool, N, C, Cse); }
    else if (img == 2) { if ((rc = se_smem_attr(se_fc_bwd_kernel<2>, smem, &a2))) return rc; se_fc_bwd_kernel<2><<<blocks, nthr, smem, st>>>(draw, pooled, Wr, br, We, be, d_e, r, d_rpre, dpool, N, C, Cse); }
    else { if ((rc = se_smem_attr(se_fc_bwd_kernel<1>, smem, &a1))) return rc; se_fc_bwd_kernel<1><<<blocks, nthr, smem, st>>>(draw, pooled, Wr, br, We, be, d_e, r, d_rpre, dpool, N, C, Cse); }
    DFD_LAUNCH_CHECK();
    return dfd_se_fc_wgrad(d_e, r, d_rpre, pooled, dWr, dbr, dWe, dbe, N, C, Cse, stream);
}

// SE parameter gradients from the per-image vectors of the backward chain (dfd_se_fc_bwd / dfd_se_bwd_chain):
// dWe += d_e^T r, dbe += sum d_e, dWr += d_rpre^T pooled, dbr += sum d_rpre   (order-deterministic)
int dfd_se_fc_wgrad(const float* d_e, const float* r, const float* d_rpre, const float* pooled, float* dWr, float* dbr,
                    float* dWe, float* dbe, int N, int C, int Cse, void* stream) {
    if (N <= 0 || C <= 0 || Cse <= 0) return dfd_set_error(DFD_ERR_ARG, "dfd_se_fc_wgrad: sizes");
    cudaStream_t st = (cudaStream_t)stream;
    // image splits: only as many as it takes to fill the GPU (the split partials are summed in order by the last block of
    // every column group: fixed slots in the library scratch, no atomics)
    const int bx = cdiv((long long)C * Cse, 128);
    int nsplit = N >= 64 ? 16 : (N >= 8 ? 4 : 1);
    while (nsplit > 1 && ((long long)bx * nsplit > 2368 || (long long)nsplit * bx * 128 * 4 > SMALL_WS_FLOATS)) nsplit >>= 1;
    if (nsplit > 1 && bx > SMALL_TICKETS) nsplit = 1;          // a single split needs no scratch at all
    se_fc_wgrad_kernel<<<dim3(bx, nsplit), 128, 0, st>>>(d_e, r, d_rpre, pooled, dWr, dbr, dWe, dbe, N, C, Cse);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_head_max_classes(void) { return HEAD_KMAX; }

int dfd_head_fwd(const float* pooled, const float* W, const float* b, float* logits, int N, int F, int K,
                 const long long* tgt_i, const float* tgt_f, float smoothing, float loss_scale,
                 const float* loss_scale_dev, float* loss_acc, float* correct_acc, float* dlogits, void* stream) {
    if (N <= 0 || F <= 0 || K <= 0) return dfd_set_error(DFD_ERR_ARG, "dfd_head_fwd: sizes");
    if (K > HEAD_KMAX) return dfd_set_error(DFD_ERR_UNSUPPORTED, "dfd_head_fwd: num_classes exceeds DFD_HEAD_KMAX (4096)");
    if (loss_acc && K < 2) return dfd_set_error(DFD_ERR_UNSUPPORTED, "dfd_head_fwd: a cross-entropy loss needs num_classes >= 2");
    if (loss_acc && !tgt_i && !tgt_f) return dfd_set_error(DFD_ERR_ARG, "dfd_head_fwd: loss without target");
    if (loss_acc && 2 * (long long)N > SMALL_WS_FLOATS) return dfd_set_error(DFD_ERR_UNSUPPORTED, "dfd_head_fwd: batch exceeds the reduction scratch");
    cudaStream_t st = (cudaStream_t)stream;
    if (K != 2) {
        int rc = head_gemm<true, true>(pooled, F, W, F, logits, K, b, 0, N, K, F, st);               // logits = pooled W^T + b
        if (rc || !loss_acc) return rc;
        head_loss_kernel<<<N, HL_THREADS, 0, st>>>(logits, K, tgt_i, tgt_f, smoothing, 1.f / (float)N, loss_scale,
                                                   loss_scale_dev, loss_acc, correct_acc, dlogits);
        DFD_LAUNCH_CHECK();
        return DFD_OK;
    }
    head_fwd_kernel<<<N, 64, 0, st>>>(pooled, W, b, logits, F, K, tgt_i, tgt_f, smoothing,
                                      1.f / (float)N, loss_scale, loss_scale_dev, loss_acc, correct_acc, dlogits);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_head_bwd(const float* dlogits, const float* pooled, const float* W, float* dW, float* db, float* dpooled,
                 int N, int F, int K, void* stream) {
    if (N <= 0 || F <= 0 || K <= 0) return dfd_set_error(DFD_ERR_ARG, "dfd_head_bwd: sizes");
    if (K > HEAD_KMAX) return dfd_set_error(DFD_ERR_UNSUPPORTED, "dfd_head_bwd: num_classes exceeds DFD_HEAD_KMAX (4096)");
    cudaStream_t st = (cudaStream_t)stream;
    if (K != 2) {
        int rc = head_gemm<true, false>(dlogits, K, W, F, dpooled, F, nullptr, 0, N, F, K, st);      // dpooled = dlogits W
        if (rc) return rc;
        rc = head_gemm<false, false>(dlogits, K, pooled, F, dW, F, nullptr, 1, K, F, N, st);         // dW += dlogits^T pooled
        if (rc) return rc;
        head_bias_grad_kernel<<<cdiv(K, 128), 128, 0, st>>>(dlogits, db, N, K);
        DFD_LAUNCH_CHECK();
        return DFD_OK;
    }
    head_dgrad_kernel<<<cdiv((long long)N * F, 256), 256, 0, st>>>(dlogits, W, dpooled, N, F, K);
    DFD_LAUNCH_CHECK();
    head_wgrad_kernel<<<dim3(cdiv((long long)K * F, 128), N >= 64 ? 16 : (N >= 8 ? 4 : 1)), 128, 0, st>>>(dlogits, pooled, dW, db, N, F, K);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

#define DISPATCH_16(dt, ...)                                          \
    if ((dt) == DFD_DT_FP16) { typedef __half T16; __VA_ARGS__; }     \
    else { typedef bf16 T16; __VA_ARGS__; }

int dfd_sgd_step(float* p, const float* g, float* m, long long n, float lr, float momentum, float wd, int nesterov,
                 float grad_scale, const float* gscale_dev, const int* skip, void* p16, int dt, const float* lr_dev,
                 void* stream) {
    if (n <= 0) return DFD_OK;
    DISPATCH_16(dt, (sgd_kernel<T16><<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, g, m, (size_t)n, lr, momentum, wd, nesterov, grad_scale, gscale_dev, skip, p16, lr_dev)));
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                  float wd, int decoupled, int step, float grad_scale, const float* gscale_dev, const int* skip, void* p16,
                  int dt, const float* lr_dev, const int* step_dev, void* stream) {
    if (n <= 0) return DFD_OK;
    float bc1 = 1.f - powf(b1, (float)step);
    float bc2s = sqrtf(1.f - powf(b2, (float)step));
    DISPATCH_16(dt, (adam_kernel<T16><<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, (size_t)n, lr, b1, b2, eps, wd, decoupled, bc1, bc2s, grad_scale, gscale_dev, skip, p16, lr_dev, step_dev)));
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_rmsprop_tf_step(float* p, const float* g, float* sq, float* mom, long long n, float lr, float alpha,
                        float eps, float wd, float momentum, float grad_scale, const float* gscale_dev, const int* skip,
                        void* p16, int dt, const float* lr_dev, void* stream) {
    if (n <= 0) return DFD_OK;
    DISPATCH_16(dt, (rmsprop_tf_kernel<T16><<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, g, sq, mom, (size_t)n, lr, alpha, eps, wd, momentum, grad_scale, gscale_dev, skip, p16, lr_dev)));
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_opt_tick(int* step_dev, const int* skip, void* stream) {
    opt_tick_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_dev, skip);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_set_floats(float* dst, int n, float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7,
                   void* stream) {
    if (n < 0 || n > 8) return dfd_set_error(DFD_ERR_ARG, "dfd_set_floats: n in [0,8]");
    F8 f = {{v0, v1, v2, v3, v4, v5, v6, v7}};
    set_floats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(dst, n, f);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_ema_update(float* ema, const float* p, long long n, long long* ema_i64, const long long* p_i64, int n_i64,
                   float decay, void* stream) {
    if (n > 0) ema_kernel<<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(ema, p, (size_t)n, decay);
    if (n_i64 > 0) ema_i64_kernel<<<cdiv(n_i64, 128), 128, 0, (cudaStream_t)stream>>>(ema_i64, p_i64, n_i64, decay);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_cast_arena(const float* p, void* p16, long long n, int dt, void* stream) {
    if (n <= 0) return DFD_OK;
    DISPATCH_16(dt, (cast_arena_kernel<T16><<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, (T16*)p16, (size_t)n)));
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_check_finite(const float* g, long long n, int* flag, void* stream) {
    if (n <= 0) return DFD_OK;
    check_finite_kernel<<<flat_blocks(n), 256, 0, (cudaStream_t)stream>>>(g, (size_t)n, flag);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

int dfd_update_loss_scale(int* flag, float* scale, int* good_steps, int interval, float* inv_scale_out, void* stream) {
    update_loss_scale_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(flag, scale, good_steps, interval, inv_scale_out);
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

// table: device array of {src, dst, O, I} (see TransposeDesc); all tensors share dtype dt
int dfd_transpose_weights(const void* table, int count, int dt, void* stream) {
    if (count <= 0) return DFD_OK;
    dim3 grid(8, 16, count), block(32, 8, 1);      // blocks beyond a tensor's 32 x 32 tiles fall through their loops
    DISPATCH_16(dt, (transpose_weights_kernel<T16><<<grid, block, 0, (cudaStream_t)stream>>>((const TransposeDesc*)table)));
    DFD_LAUNCH_CHECK();
    return DFD_OK;
}

}  // extern "C"
