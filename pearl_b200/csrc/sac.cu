// sac.cu — continuous Soft Actor-Critic learner (ContinuousSoftActorCritic.learn_batch driven by
// PolicyLearner.learn), replacing
//   policy_learners/sequential_decision_making/actor_critic_base.py:309-366   (actor step, critic step, soft update)
//   policy_learners/sequential_decision_making/soft_actor_critic_continuous.py:131-231 (losses, entropy autotune)
//   neural_networks/sequential_decision_making/actor_networks.py:29-51,488-591 (GaussianActorNetwork.sample_action)
//   neural_networks/sequential_decision_making/twin_critic.py:75-91, q_value_networks.py:152-174
//   utils/functional_utils/learning/critic_utils.py:103-122,170-203, torch.optim.AdamW(amsgrad=True)
//
// Round-1 structure: the step is a fixed sequence of launches of ONE generic tiled fp32 contraction
// kernel (forward y = act(x W^T + b), backward-data dx = dy W (* relu mask), backward-weight
// dW = dy^T x with the bias gradient as an implicit ones column; the state||action concat and the twin
// critics are handled inside the kernel: two-source operands, blockIdx.z = critic) plus small
// elementwise kernels for the tanh-Gaussian policy, the losses and AdamW.  fp32, fixed summation
// order (deterministic).  The tensor-core path of the DQN learner is not applied here yet.
#include <math.h>
#include <stdarg.h>

#include <new>

#include "common.cuh"
#include "gemm.cuh"

using namespace prl;

namespace {

// per-call pointers the captured round reads through (the graph itself never changes between calls)
struct SacCall {
    const float *noise;      // [rounds][2][B][A]
    const int32_t *slots;    // [rounds][B]
    float *out_actor, *out_critic, *out_entropy;
};

// ------------------------------------------------------------------ elementwise pieces
// batch rows of one round from the replay ring
__global__ void k_sac_gather(const uint32_t *__restrict__ records, prl_buf_layout L, int obs, int act, const SacCall *__restrict__ call,
                             const int *__restrict__ round_idx, int B, float *__restrict__ S, float *__restrict__ A, float *__restrict__ R,
                             float *__restrict__ S2, float *__restrict__ T) {
    const int lane = threadIdx.x & 31, w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= B) return;
    const int32_t *slots = call->slots + (size_t)(*round_idx) * B;
    const uint32_t *r = records + (size_t)slots[w] * L.record_words;
    for (int p = lane; p < obs; p += 32) {
        S[(size_t)w * obs + p] = __uint_as_float(r[L.off_state + p]);
        S2[(size_t)w * obs + p] = __uint_as_float(r[L.off_next_state + p]);
    }
    for (int p = lane; p < act; p += 32) A[(size_t)w * act + p] = __uint_as_float(r[L.off_action + p]);
    if (lane == 0) { R[w] = __uint_as_float(r[L.off_reward]); T[w] = (r[L.off_flags] & 1u) ? 1.f : 0.f; }
}

// GaussianActorNetwork.sample_action (actor_networks.py:551-591) with the rsample noise given
__global__ void k_sac_sample(int B, int A, const float *__restrict__ mean, const float *__restrict__ z, const SacCall *__restrict__ call,
                             const int *__restrict__ round_idx, int which, const float *__restrict__ low, const float *__restrict__ high,
                             float *__restrict__ action, float *__restrict__ na_out, float *__restrict__ std_out, float *__restrict__ logp) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float *noise = call->noise + (size_t)(2 * (*round_idx) + which) * B * A;
    float lp = 0.f;
    for (int d = 0; d < A; d++) {
        const size_t o = (size_t)b * A + d;
        const float log_std = -5.f + 3.5f * (tanhf(z[o]) + 1.f);
        const float sd = expf(log_std), eps = noise[o];
        const float sample = mean[o] + sd * eps;
        const float na = tanhf(sample);
        const float lo = low[d], hi = high[d], bound = (hi - lo) * 0.5f;
        action[o] = (((hi - lo) * (na + 1.0f)) / 2.f) + lo;
        na_out[o] = na; std_out[o] = sd;
        const float diff = sample - mean[o];
        float t = -(diff * diff) / (2.f * sd * sd) - log_std - 0.91893853320467274178f;   // Normal.log_prob
        t -= logf(bound * (1.f - na * na) + 1e-6f);
        lp += t;
    }
    logp[b] = lp;
}

// actor loss = mean(alpha * logp - min(q1, q2)); routes -1/B to the smaller critic
__global__ void k_sac_actor_loss(int B, const float *__restrict__ q, const float *__restrict__ logp, const float *__restrict__ alpha,
                                 float *__restrict__ dq, const SacCall *__restrict__ call, const int *__restrict__ round_idx) {
    __shared__ float red[256];
    float s = 0.f;
    const float al = *alpha, ib = 1.f / (float)B;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const float q1 = q[b], q2 = q[B + b];
        const bool first = q1 <= q2;
        s += al * logp[b] - (first ? q1 : q2);
        dq[b] = first ? -ib : 0.f;
        dq[B + b] = first ? 0.f : -ib;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) call->out_actor[*round_idx] = red[0] * ib;
}

// gradients of the actor loss w.r.t. the two heads (mean, pre-tanh log-std z)
__global__ void k_sac_head_grads(int B, int A, const float *__restrict__ da /* [2][B][A] from both critics */,
                                 const float *__restrict__ na, const float *__restrict__ sd, const SacCall *__restrict__ call,
                                 const int *__restrict__ round_idx, const float *__restrict__ z, const float *__restrict__ low,
                                 const float *__restrict__ high, const float *__restrict__ alpha, float *__restrict__ dmean,
                                 float *__restrict__ dz) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * A) return;
    const float *noise = call->noise + (size_t)(2 * (*round_idx)) * B * A;
    const int d = e % A;
    const float al_b = *alpha / (float)B;
    const float lo = low[d], hi = high[d], bound = (hi - lo) * 0.5f;
    const float n = na[e];
    const float dact = da[e] + da[(size_t)B * A + e];
    // d/dna: action scaling, and -log(bound (1 - na^2) + 1e-6) inside log-prob
    const float dna = dact * (hi - lo) * 0.5f + al_b * (2.f * bound * n) / (bound * (1.f - n * n) + 1e-6f);
    const float du = dna * (1.f - n * n);                      // through tanh
    dmean[e] = du;
    const float dlogstd = du * sd[e] * noise[e] - al_b;         // sample = mean + std*eps ; -log_std term of log-prob
    const float tz = tanhf(z[e]);
    dz[e] = dlogstd * 3.5f * (1.f - tz * tz);
}

// y = (min(q1t, q2t) - alpha * logp') * gamma * (1 - terminated) + reward;  dq_i = (q_i - y) / B ; critic loss
__global__ void k_sac_target(int B, const float *__restrict__ qt, const float *__restrict__ logp2, const float *__restrict__ alpha,
                             float gamma, const float *__restrict__ term, const float *__restrict__ rew, float *__restrict__ y) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float nq = fminf(qt[b], qt[B + b]) - (*alpha) * logp2[b];
    y[b] = __fadd_rn(__fmul_rn(__fmul_rn(nq, gamma), 1.f - term[b]), rew[b]);
}
__global__ void k_sac_critic_loss(int B, const float *__restrict__ q, const float *__restrict__ y, float *__restrict__ dq,
                                  const SacCall *__restrict__ call, const int *__restrict__ round_idx) {
    const float loss = twin_mse_block(B, q, y, dq);
    if (threadIdx.x == 0) call->out_critic[*round_idx] = loss;
}

// entropy coefficient: loss = mean(-exp(log_alpha) * (logp + target_entropy)); AdamW on the scalar; alpha = exp(log_alpha)
__global__ void k_sac_alpha(int B, const float *__restrict__ logp, float target_entropy, float *__restrict__ log_alpha /* [4]: w m v vmax */,
                            float *__restrict__ alpha, AdamHp h, const float2 *__restrict__ scal, const int *__restrict__ round_idx,
                            const SacCall *__restrict__ call, int autotune) {
    __shared__ float red[256];
    if (!autotune) {                       // fixed entropy coefficient: only the round counter advances
        if (threadIdx.x == 0) *const_cast<int *>(round_idx) += 1;
        return;
    }
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) s += logp[b] + target_entropy;
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) {
        const float mean = red[0] / (float)B, ea = expf(log_alpha[0]);
        call->out_entropy[*round_idx] = -ea * mean;
        const float g = -ea * mean;                 // d/dlog_alpha
        const float2 sc = scal[*round_idx];
        float mm = log_alpha[1], vv = log_alpha[2], xx = log_alpha[3];
        const float p = adamw1(log_alpha[0], mm, vv, xx, g, h, sc.x, sc.y);
        log_alpha[0] = p; log_alpha[1] = mm; log_alpha[2] = vv; log_alpha[3] = xx;
        *alpha = expf(p);
        *const_cast<int *>(round_idx) += 1;
    }
}

}  // namespace

// ------------------------------------------------------------------ host side
struct prl_sac {
    prl_sac_cfg cfg;
    int Pa, Pc;                       // actor parameters; parameters of ONE critic
    // actor layout offsets
    int aW1, ab1, aW2, ab2, aWmu, abmu, aWsd, absd;
    int cW1, cb1, cW2, cb2, cW3, cb3; // critic layout offsets (within one critic)
    float *actor, *actor_m, *actor_v, *actor_x;
    float *critic, *critic_m, *critic_v, *critic_x, *critic_t;
    float *log_alpha, *alpha;         // log_alpha[4] = value, m, v, vmax ; alpha scalar
    const float *low, *high;
    int64_t adam_step;
    // workspace
    float *S, *A, *R, *S2, *T, *h1, *h2, *mean, *z, *act_s, *na, *sd, *logp, *logp2, *c1, *c2, *q, *qt, *dq, *dc2, *dc1, *da, *dmean, *dz,
        *dh2, *dh1, *y, *g_actor, *g_critic;
    int32_t *slots, *logical;
    float2 *scal_a, *scal_c;
    SacCall *call;
    int *round_idx;
    bool use_graph;
    cudaGraphExec_t graph_exec;
    int graph_batch;
    const uint32_t *graph_buf;
    int launches_per_round;
    float2 *scal_host[2];
    cudaEvent_t scal_done[2];
    int scal_next;
    int64_t last_launches;
};

static int64_t al64(int64_t x) { return (x + 255) / 256 * 256; }

static void sac_layout(prl_sac *s) {
    const prl_sac_cfg &c = s->cfg;
    int o = 0;
    s->aW1 = o; o += c.actor_h1 * c.obs_dim; s->ab1 = o; o += c.actor_h1;
    s->aW2 = o; o += c.actor_h2 * c.actor_h1; s->ab2 = o; o += c.actor_h2;
    s->aWmu = o; o += c.act_dim * c.actor_h2; s->abmu = o; o += c.act_dim;
    s->aWsd = o; o += c.act_dim * c.actor_h2; s->absd = o; o += c.act_dim;
    s->Pa = o;
    const int D = c.obs_dim + c.act_dim;
    o = 0;
    s->cW1 = o; o += c.critic_h1 * D; s->cb1 = o; o += c.critic_h1;
    s->cW2 = o; o += c.critic_h2 * c.critic_h1; s->cb2 = o; o += c.critic_h2;
    s->cW3 = o; o += c.critic_h2; s->cb3 = o; o += 1;
    s->Pc = o;
}

static int sac_check(const prl_sac_cfg *c) {
    PRL_REQUIRE(c, "null cfg");
    PRL_REQUIRE(c->obs_dim > 0 && c->act_dim > 0 && c->actor_h1 > 0 && c->actor_h2 > 0 && c->critic_h1 > 0 && c->critic_h2 > 0,
                "dimensions must be positive");
    PRL_REQUIRE(c->max_batch > 0 && c->max_rounds > 0, "max_batch / max_rounds must be positive");
    return PRL_OK;
}

extern "C" int64_t prl_sac_actor_param_count(const prl_sac_cfg *c) {
    if (sac_check(c)) return -1;
    prl_sac t; t.cfg = *c; sac_layout(&t);
    return t.Pa;
}
extern "C" int64_t prl_sac_critic_param_count(const prl_sac_cfg *c) {   // ONE critic; the twin vector holds two
    if (sac_check(c)) return -1;
    prl_sac t; t.cfg = *c; sac_layout(&t);
    return t.Pc;
}

struct SacWs { int64_t off[40]; int64_t total; };
static SacWs sac_ws(const prl_sac_cfg *c, int Pa, int Pc) {
    SacWs w; int64_t o = 0; int k = 0;
    const int64_t B = c->max_batch, A = c->act_dim, O = c->obs_dim;
    auto add = [&](int64_t floats) { w.off[k++] = o; o = al64(o + floats * 4); };
    add(B * O); add(B * A); add(B); add(B * O); add(B);                                  // S A R S2 T
    add(B * c->actor_h1); add(B * c->actor_h2); add(B * A); add(B * A);                   // h1 h2 mean z
    add(B * A); add(B * A); add(B * A); add(B); add(B);                                  // act_s na sd logp logp2
    add(2 * B * c->critic_h1); add(2 * B * c->critic_h2); add(2 * B); add(2 * B);         // c1 c2 q qt
    add(2 * B); add(2 * B * c->critic_h2); add(2 * B * c->critic_h1); add(2 * B * A);     // dq dc2 dc1 da
    add(B * A); add(B * A); add(B * c->actor_h2); add(B * c->actor_h1); add(B);          // dmean dz dh2 dh1 y
    add(Pa); add(2 * (int64_t)Pc);                                                        // g_actor g_critic
    add((int64_t)c->max_rounds * B); add((int64_t)c->max_rounds * B);                    // slots logical (int32)
    add(4 * (int64_t)c->max_rounds + 64);                                                 // scal_a | scal_c | call | round_idx
    w.total = o;
    return w;
}
extern "C" int64_t prl_sac_workspace_bytes(const prl_sac_cfg *c) {
    if (sac_check(c)) return -1;
    prl_sac t; t.cfg = *c; sac_layout(&t);
    return sac_ws(c, t.Pa, t.Pc).total;
}

extern "C" int prl_sac_create(prl_sac **out, const prl_sac_cfg *cfg, float *actor_w, float *actor_m, float *actor_v, float *actor_vmax,
                              float *critic_w, float *critic_m, float *critic_v, float *critic_vmax, float *critic_target_w,
                              float *log_alpha4, float *alpha1, const float *low_dev, const float *high_dev, int64_t adam_step,
                              void *workspace) {
    PRL_REQUIRE(out && actor_w && actor_m && actor_v && actor_vmax && critic_w && critic_m && critic_v && critic_vmax &&
                    critic_target_w && log_alpha4 && alpha1 && low_dev && high_dev && workspace, "null argument");
    int rc = sac_check(cfg);
    if (rc) return rc;
    prl_sac *s = new (std::nothrow) prl_sac();
    if (!s) return fail(PRL_ENOMEM, "out of host memory");
    s->cfg = *cfg;
    sac_layout(s);
    s->actor = actor_w; s->actor_m = actor_m; s->actor_v = actor_v; s->actor_x = actor_vmax;
    s->critic = critic_w; s->critic_m = critic_m; s->critic_v = critic_v; s->critic_x = critic_vmax; s->critic_t = critic_target_w;
    s->log_alpha = log_alpha4; s->alpha = alpha1; s->low = low_dev; s->high = high_dev;
    s->adam_step = adam_step;
    SacWs w = sac_ws(cfg, s->Pa, s->Pc);
    char *b = (char *)workspace;
    float **f[] = {&s->S, &s->A, &s->R, &s->S2, &s->T, &s->h1, &s->h2, &s->mean, &s->z, &s->act_s, &s->na, &s->sd, &s->logp, &s->logp2,
                   &s->c1, &s->c2, &s->q, &s->qt, &s->dq, &s->dc2, &s->dc1, &s->da, &s->dmean, &s->dz, &s->dh2, &s->dh1, &s->y,
                   &s->g_actor, &s->g_critic};
    int k = 0;
    for (auto p : f) *p = (float *)(b + w.off[k++]);
    s->slots = (int32_t *)(b + w.off[k++]); s->logical = (int32_t *)(b + w.off[k++]);
    s->scal_a = (float2 *)(b + w.off[k++]); s->scal_c = s->scal_a + cfg->max_rounds;
    s->call = (SacCall *)(s->scal_c + cfg->max_rounds); s->round_idx = (int *)(s->call + 1);
    s->scal_next = 0; s->use_graph = true; s->graph_exec = nullptr; s->graph_batch = 0; s->graph_buf = nullptr; s->last_launches = 0;
    static_assert(sizeof(SacCall) + 4 <= 64 * 4, "call block fits the reserved tail");
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 2 && e == cudaSuccess; i++) {
        e = cudaHostAlloc((void **)&s->scal_host[i], (size_t)cfg->max_rounds * 16 + 256, cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->scal_done[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { delete s; return fail(PRL_ECUDA, "prl_sac_create: %s", cudaGetErrorString(e)); }
    *out = s;
    return PRL_OK;
}
extern "C" int prl_sac_destroy(prl_sac *s) {
    if (!s) return PRL_OK;
    for (int i = 0; i < 2; i++) { cudaEventSynchronize(s->scal_done[i]); cudaEventDestroy(s->scal_done[i]); cudaFreeHost(s->scal_host[i]); }
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    delete s;
    return PRL_OK;
}
extern "C" int64_t prl_sac_adam_step(const prl_sac *s) { return s ? s->adam_step : -1; }

// one learner round, launched (or captured) on `st`; everything round-dependent is read on the device through
// s->call / s->round_idx
static int sac_round(prl_sac *s, prl_buf *buf, int B, cudaStream_t st) {
    const prl_sac_cfg &c = s->cfg;
    const int O = c.obs_dim, A = c.act_dim, D = O + A;
    const int H1 = c.actor_h1, H2 = c.actor_h2, C1 = c.critic_h1, C2 = c.critic_h2;
    const long long Pc = s->Pc;
    AdamHp ha{(float)(1.0 - c.actor_lr * c.weight_decay), (float)(1.0 - c.beta1), (float)c.beta2, (float)(1.0 - c.beta2), (float)c.eps};
    AdamHp hc{(float)(1.0 - c.critic_lr * c.weight_decay), (float)(1.0 - c.beta1), (float)c.beta2, (float)(1.0 - c.beta2), (float)c.eps};
    GemmLauncher L; L.st = st;
    const float *aw = s->actor, *cw = s->critic, *ct = s->critic_t;
    const long long sC1 = (long long)B * C1, sC2 = (long long)B * C2;
    auto actor_forward = [&](const float *X) {
        L.fwd(mat(X, O), B, aw + s->aW1, O, 0, aw + s->ab1, 0, H1, O, true, s->h1, H1, 0);
        L.fwd(mat(s->h1, H1), B, aw + s->aW2, H1, 0, aw + s->ab2, 0, H2, H1, true, s->h2, H2, 0);
        L.fwd(mat(s->h2, H2), B, aw + s->aWmu, H2, 0, aw + s->abmu, 0, A, H2, false, s->mean, A, 0);
        L.fwd(mat(s->h2, H2), B, aw + s->aWsd, H2, 0, aw + s->absd, 0, A, H2, false, s->z, A, 0);
    };
    auto critic_forward = [&](const float *net, const float *X, const float *Act, float *qout) {   // both critics (blockIdx.z)
        L.fwd(mat2(X, O, O, Act, A), B, net + s->cW1, D, Pc, net + s->cb1, Pc, C1, D, true, s->c1, C1, sC1, 2);
        L.fwd(mat(s->c1, C1, sC1), B, net + s->cW2, C1, Pc, net + s->cb2, Pc, C2, C1, true, s->c2, C2, sC2, 2);
        L.fwd(mat(s->c2, C2, sC2), B, net + s->cW3, C2, Pc, net + s->cb3, Pc, 1, C2, false, qout, 1, B, 2);
    };
    const int eb = 256;
    int small = 0;
    k_sac_gather<<<(B * 32 + eb - 1) / eb, eb, 0, st>>>(buf->records, buf->lay, O, A, s->call, s->round_idx, B, s->S, s->A, s->R, s->S2, s->T);
    // ---------------- actor step (actor_critic_base.py:333-343)
    actor_forward(s->S);
    k_sac_sample<<<(B + 127) / 128, 128, 0, st>>>(B, A, s->mean, s->z, s->call, s->round_idx, 0, s->low, s->high, s->act_s, s->na, s->sd, s->logp);
    critic_forward(cw, s->S, s->act_s, s->q);
    k_sac_actor_loss<<<1, 256, 0, st>>>(B, s->q, s->logp, s->alpha, s->dq, s->call, s->round_idx);
    {   // dQ/d(action) through both critics
        dim3 g2((B * C2 + eb - 1) / eb, 1, 2);
        k_head_bwd<<<g2, eb, 0, st>>>(B, C2, s->dq, cw + s->cW3, Pc, s->c2, s->dc2);
        L.bwd_x(s->dc2, C2, sC2, B, C2, cw + s->cW2, C1, Pc, 0, C1, s->dc1, C1, sC1, s->c1, C1, sC1, false, 2);
        L.bwd_x(s->dc1, C1, sC1, B, C1, cw + s->cW1, D, Pc, O, A, s->da, A, (long long)B * A, nullptr, 0, 0, false, 2);
    }
    k_sac_head_grads<<<(B * A + eb - 1) / eb, eb, 0, st>>>(B, A, s->da, s->na, s->sd, s->call, s->round_idx, s->z, s->low, s->high, s->alpha,
                                                         s->dmean, s->dz);
    {   // actor backward
        float *ga = s->g_actor;
        L.bwd_w(s->dmean, A, 0, B, A, mat(s->h2, H2), H2, ga + s->aWmu, H2, 0, ga + s->abmu, 0);
        L.bwd_w(s->dz, A, 0, B, A, mat(s->h2, H2), H2, ga + s->aWsd, H2, 0, ga + s->absd, 0);
        L.bwd_x(s->dmean, A, 0, B, A, aw + s->aWmu, H2, 0, 0, H2, s->dh2, H2, 0, nullptr, 0, 0, false);
        L.bwd_x(s->dz, A, 0, B, A, aw + s->aWsd, H2, 0, 0, H2, s->dh2, H2, 0, s->h2, H2, 0, true);
        L.bwd_w(s->dh2, H2, 0, B, H2, mat(s->h1, H1), H1, ga + s->aW2, H1, 0, ga + s->ab2, 0);
        L.bwd_x(s->dh2, H2, 0, B, H2, aw + s->aW2, H1, 0, 0, H1, s->dh1, H1, 0, s->h1, H1, 0, false);
        L.bwd_w(s->dh1, H1, 0, B, H1, mat(s->S, O), O, ga + s->aW1, O, 0, ga + s->ab1, 0);
        k_adamw<<<(s->Pa + eb - 1) / eb, eb, 0, st>>>(s->Pa, s->actor, s->actor_m, s->actor_v, s->actor_x, ga, ha, s->scal_a, s->round_idx, nullptr, 0.f, 0.f);
    }
    // ---------------- critic step with the UPDATED actor (:345-349; soft_actor_critic_continuous.py:155-205)
    actor_forward(s->S2);
    k_sac_sample<<<(B + 127) / 128, 128, 0, st>>>(B, A, s->mean, s->z, s->call, s->round_idx, 1, s->low, s->high, s->act_s, s->na, s->sd, s->logp2);
    critic_forward(ct, s->S2, s->act_s, s->qt);
    k_sac_target<<<(B + eb - 1) / eb, eb, 0, st>>>(B, s->qt, s->logp2, s->alpha, (float)c.gamma, s->T, s->R, s->y);
    critic_forward(cw, s->S, s->A, s->q);
    k_sac_critic_loss<<<1, 256, 0, st>>>(B, s->q, s->y, s->dq, s->call, s->round_idx);
    {
        float *gc = s->g_critic;
        L.bwd_w(s->dq, 1, B, B, 1, mat(s->c2, C2, sC2), C2, gc + s->cW3, C2, Pc, gc + s->cb3, Pc, 2);
        dim3 g2((B * C2 + eb - 1) / eb, 1, 2);
        k_head_bwd<<<g2, eb, 0, st>>>(B, C2, s->dq, cw + s->cW3, Pc, s->c2, s->dc2);
        L.bwd_w(s->dc2, C2, sC2, B, C2, mat(s->c1, C1, sC1), C1, gc + s->cW2, C1, Pc, gc + s->cb2, Pc, 2);
        L.bwd_x(s->dc2, C2, sC2, B, C2, cw + s->cW2, C1, Pc, 0, C1, s->dc1, C1, sC1, s->c1, C1, sC1, false, 2);
        L.bwd_w(s->dc1, C1, sC1, B, C1, mat2(s->S, O, O, s->A, A), D, gc + s->cW1, D, Pc, gc + s->cb1, Pc, 2);
        const int n2p = 2 * s->Pc;
        k_adamw<<<(n2p + eb - 1) / eb, eb, 0, st>>>(n2p, s->critic, s->critic_m, s->critic_v, s->critic_x, gc, hc, s->scal_c, s->round_idx,
                                                  s->critic_t, (float)c.tau, (float)(1.0 - c.tau));
    }
    small = 12;
    // ---------------- entropy coefficient (soft_actor_critic_continuous.py:134-147); also advances the round counter
    k_sac_alpha<<<1, 256, 0, st>>>(B, s->logp, -(float)A, s->log_alpha, s->alpha, hc, s->scal_c, s->round_idx, s->call, c.autotune);
    s->launches_per_round = L.count + small;
    return PRL_OK;
}

extern "C" int prl_sac_learn(prl_sac *s, prl_buf *buf, int rounds, int batch, const float *noise_dev, float *out_actor_loss,
                             float *out_critic_loss, float *out_entropy_loss, int32_t *out_logical, void *stream_) {
    PRL_REQUIRE(s && buf && noise_dev && out_actor_loss && out_critic_loss && out_entropy_loss, "null argument");
    const prl_sac_cfg &c = s->cfg;
    PRL_REQUIRE(rounds > 0 && rounds <= c.max_rounds && batch > 0 && batch <= c.max_batch, "rounds / batch outside the configured maxima");
    PRL_REQUIRE((buf->desc.flags & PRL_BUF_CONTINUOUS) && buf->desc.obs_dim == c.obs_dim && buf->desc.act_dim == c.act_dim,
                "SAC needs a continuous-action buffer with matching dimensions");
    cudaStream_t st = (cudaStream_t)stream_;
    int rc = prl_buf_sample_indices(buf, rounds, batch, out_logical ? out_logical : s->logical, s->slots, stream_);
    if (rc) return rc;
    // per-call block: AdamW scalars of every round (actor lr / critic lr, as torch evaluates them in double) + pointers
    const int sb = s->scal_next; s->scal_next ^= 1;
    PRL_CUDA(cudaEventSynchronize(s->scal_done[sb]));
    float2 *hs = s->scal_host[sb];
    for (int r = 0; r < rounds; r++) {
        const double step = (double)(s->adam_step + r + 1);
        const double bc1 = 1.0 - pow(c.beta1, step), bc2 = 1.0 - pow(c.beta2, step);
        hs[r] = make_float2((float)(c.actor_lr / bc1), (float)sqrt(bc2));
        hs[c.max_rounds + r] = make_float2((float)(c.critic_lr / bc1), (float)sqrt(bc2));
    }
    SacCall *hc = reinterpret_cast<SacCall *>(hs + 2 * (size_t)c.max_rounds);
    hc->noise = noise_dev; hc->slots = s->slots; hc->out_actor = out_actor_loss; hc->out_critic = out_critic_loss; hc->out_entropy = out_entropy_loss;
    int *hround = reinterpret_cast<int *>(hc + 1);
    *hround = 0;
    // scal_a | scal_c | call | round_idx are contiguous on the device in the same order
    PRL_CUDA(cudaMemcpyAsync(s->scal_a, hs, 2 * (size_t)c.max_rounds * 8 + sizeof(SacCall) + 4, cudaMemcpyHostToDevice, st));
    PRL_CUDA(cudaEventRecord(s->scal_done[sb], st));

    if (s->use_graph) {
        if (!s->graph_exec || s->graph_batch != batch || s->graph_buf != buf->records) {
            if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
            cudaStream_t cs;
            PRL_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t graph = nullptr;
            cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                sac_round(s, buf, batch, cs);
                e = cudaStreamEndCapture(cs, &graph);
            }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&s->graph_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            cudaStreamDestroy(cs);
            if (e != cudaSuccess) { s->graph_exec = nullptr; return fail(PRL_ECUDA, "prl_sac_learn: graph capture failed: %s", cudaGetErrorString(e)); }
            s->graph_batch = batch; s->graph_buf = buf->records;
        }
        for (int r = 0; r < rounds; r++) PRL_CUDA(cudaGraphLaunch(s->graph_exec, st));
    } else {
        for (int r = 0; r < rounds; r++) {
            rc = sac_round(s, buf, batch, st);
            if (rc) return rc;
        }
    }
    PRL_CUDA(cudaGetLastError());
    s->adam_step += rounds;
    s->last_launches = s->launches_per_round * rounds;
    return PRL_OK;
}
extern "C" int prl_sac_set_graph(prl_sac *s, int enable) {
    PRL_REQUIRE(s, "null handle");
    s->use_graph = enable != 0;
    return PRL_OK;
}
extern "C" int64_t prl_sac_last_launches(const prl_sac *s) { return s ? s->last_launches : -1; }
