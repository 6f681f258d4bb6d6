// dsac.cu — discrete Soft Actor-Critic learner (SoftActorCritic.learn_batch driven by PolicyLearner.learn), replacing
//   policy_learners/policy_learner.py:162-204                                   (training_rounds x sample + learn_batch)
//   policy_learners/sequential_decision_making/actor_critic_base.py:309-366     (actor step, critic step, soft update)
//   policy_learners/sequential_decision_making/soft_actor_critic.py:151-286     (losses, entropy autotune)
//   neural_networks/sequential_decision_making/actor_networks.py:107-153        (VanillaActorNetwork, softmax head)
//   neural_networks/sequential_decision_making/twin_critic.py:75-91, q_value_networks.py:152-174
//   utils/functional_utils/learning/critic_utils.py:103-122,170-203, torch.optim.AdamW(amsgrad=True), torch.optim.Adam
//
// A round is a fixed launch sequence (captured once per (batch, buffer) into a CUDA graph and replayed): the dense layers
// are the generic contraction of gemm.cuh (twin critics along blockIdx.z, state || one-hot action as a two-source operand),
// plus small kernels for the softmax policy, the losses and the optimizers.  The step takes expectations over the softmax
// policy instead of sampling, so it draws no random numbers.  Q(s, a) for EVERY action a (actor loss on s, target on s')
// folds the one-hot input into the first layer: relu(s W1[:, :obs]^T + W1[:, obs + a] + b1), the state product computed
// once per row and expanded to B x A rows.  Every round-dependent scalar (AdamW lr / bias corrections / decay, the
// entropy Adam step) is read from the per-call device block, so a replayed graph follows learning-rate changes.
// fp32, fixed summation orders (deterministic).
#include <math.h>

#include <new>

#include "common.cuh"
#include "gemm.cuh"

using namespace prl;

namespace {

// per-round optimizer scalars, filled on the host for every learn() call
struct DsacScal {
    float a_ss, a_bc2s, a_decay;   // actor AdamW: lr / bc1, sqrt(bc2), 1 - lr * weight_decay
    float c_ss, c_bc2s, c_decay;   // critics
    float e_ss, e_bc2s;            // entropy Adam: lr / bc1, sqrt(bc2)
};
// per-call pointers the captured round reads through
struct DsacCall {
    const int32_t *slots;          // [rounds][B]
    float *out_actor, *out_critic, *out_entropy;
};

// batch rows of one round from the replay ring; the taken action as an id and as a one-hot row
__global__ void k_dsac_gather(const uint32_t *__restrict__ records, prl_buf_layout L, int obs, int A, const DsacCall *__restrict__ call,
                              const int *__restrict__ round_idx, int B, float *__restrict__ S, float *__restrict__ S2,
                              float *__restrict__ onehot, float *__restrict__ R, float *__restrict__ T) {
    const int lane = threadIdx.x & 31, w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= B) return;
    const int32_t *slots = call->slots + (size_t)(*round_idx) * B;
    const uint32_t *r = records + (size_t)slots[w] * L.record_words;
    for (int p = lane; p < obs; p += 32) {
        S[(size_t)w * obs + p] = __uint_as_float(r[L.off_state + p]);
        S2[(size_t)w * obs + p] = __uint_as_float(r[L.off_next_state + p]);
    }
    const int a = (int32_t)r[L.off_action];
    for (int p = lane; p < A; p += 32) onehot[(size_t)w * A + p] = p == a ? 1.f : 0.f;
    if (lane == 0) { R[w] = __uint_as_float(r[L.off_reward]); T[w] = (r[L.off_flags] & 1u) ? 1.f : 0.f; }
}

// the one-hot fold: H1[z][b * A + a][j] = relu(P[z][b][j] + W1[z][j][obs + a] + b1[z][j]), P = s W1[:, :obs]^T
__global__ void k_dsac_expand(int B, int A, int C1, int obs, const float *__restrict__ P, const float *__restrict__ w1,
                              const float *__restrict__ b1, long long net_stride, float *__restrict__ H1) {
    const int z = blockIdx.z;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)B * A * C1) return;
    const int j = (int)(e % C1);
    const long long row = e / C1;
    const int b = (int)(row / A), a = (int)(row % A);
    const float *w = w1 + z * net_stride, *bb = b1 + z * net_stride;
    const float v = P[(size_t)z * B * C1 + (size_t)b * C1 + j] + __ldg(w + (size_t)j * (obs + A) + obs + a) + __ldg(bb + j);
    H1[(size_t)z * B * A * C1 + e] = fmaxf(v, 0.f);
}

__device__ __forceinline__ float row_max(const float *l, int A) {
    float mx = l[0];
    for (int a = 1; a < A; a++) mx = fmaxf(mx, l[a]);
    return mx;
}

// actor loss (soft_actor_critic.py:247-286): p = softmax(logits), q = min(Q1, Q2)(s, .),
// loss = mean_{B x A}(p (alpha log(p + 1e-8) - q)); dlogits = p (g - sum p g), g = dloss/dp; ent[b] = sum_a p log(p + 1e-8)
__global__ void k_dsac_actor_loss(int B, int A, const float *__restrict__ logits, const float *__restrict__ qall,
                                  const float *__restrict__ alpha, float *__restrict__ dlogits, float *__restrict__ ent,
                                  const DsacCall *__restrict__ call, const int *__restrict__ round_idx) {
    __shared__ float red[256];
    const float al = *alpha, inv = 1.f / (float)(B * A);
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const float *l = logits + (size_t)b * A, *q1 = qall + (size_t)b * A, *q2 = qall + (size_t)B * A + (size_t)b * A;
        const float mx = row_max(l, A);
        float sum = 0.f;
        for (int a = 0; a < A; a++) sum += expf(l[a] - mx);
        float row = 0.f, e = 0.f, pg = 0.f;
        for (int a = 0; a < A; a++) {
            const float p = expf(l[a] - mx) / sum, lp = logf(p + 1e-8f), q = fminf(q1[a], q2[a]);
            row += p * (al * lp - q);
            e += p * lp;
            const float g = (al * lp - q + al * p / (p + 1e-8f)) * inv;
            dlogits[(size_t)b * A + a] = g;
            pg += p * g;
        }
        for (int a = 0; a < A; a++) {
            const float p = expf(l[a] - mx) / sum;
            dlogits[(size_t)b * A + a] = p * (dlogits[(size_t)b * A + a] - pg);
        }
        ent[b] = e;
        s += row;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) call->out_actor[*round_idx] = red[0] * inv;
}

// critic target (soft_actor_critic.py:180-245): V(s') = sum_a p'(min(Q1t, Q2t)(s', a) - alpha log(p' + 1e-8)),
// y = V(s') gamma (1 - terminated) + r
__global__ void k_dsac_target(int B, int A, const float *__restrict__ logits, const float *__restrict__ qtall,
                              const float *__restrict__ alpha, float gamma, const float *__restrict__ term, const float *__restrict__ rew,
                              float *__restrict__ y) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float al = *alpha;
    const float *l = logits + (size_t)b * A, *q1 = qtall + (size_t)b * A, *q2 = qtall + (size_t)B * A + (size_t)b * A;
    const float mx = row_max(l, A);
    float sum = 0.f;
    for (int a = 0; a < A; a++) sum += expf(l[a] - mx);
    float v = 0.f;
    for (int a = 0; a < A; a++) {
        const float p = expf(l[a] - mx) / sum;
        v += (fminf(q1[a], q2[a]) - al * logf(p + 1e-8f)) * p;
    }
    y[b] = __fadd_rn(__fmul_rn(__fmul_rn(v, gamma), 1.f - term[b]), rew[b]);
}

__global__ void k_dsac_critic_loss(int B, const float *__restrict__ q, const float *__restrict__ y, float *__restrict__ dq,
                                   const DsacCall *__restrict__ call, const int *__restrict__ round_idx) {
    const float loss = twin_mse_block(B, q, y, dq);
    if (threadIdx.x == 0) call->out_critic[*round_idx] = loss;
}

// AdamW(amsgrad) over a flat vector with this round's scalars (which = 0: actor, 1: critics) from the per-call block;
// optional soft update of a target vector with the NEW parameters (critic_utils.py:103-122)
__global__ void k_dsac_adamw(int n, float *__restrict__ w, float *__restrict__ m, float *__restrict__ v, float *__restrict__ vmax,
                             const float *__restrict__ grad, AdamHp h, const DsacScal *__restrict__ scal, int which,
                             const int *__restrict__ round_idx, float *__restrict__ target, float tau, float omtau) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const DsacScal sc = scal[*round_idx];
    h.decay = which ? sc.c_decay : sc.a_decay;
    float mm = m[i], vv = v[i], xx = vmax[i];
    const float p = adamw1(w[i], mm, vv, xx, grad[i], h, which ? sc.c_ss : sc.a_ss, which ? sc.c_bc2s : sc.a_bc2s);
    w[i] = p; m[i] = mm; v[i] = vv; vmax[i] = xx;
    if (target) target[i] = __fadd_rn(__fmul_rn(tau, p), __fmul_rn(omtau, target[i]));
}

// entropy coefficient (soft_actor_critic.py:151-178): H = -mean_b ent[b]; loss = exp(log_alpha) (H - target_entropy);
// torch.optim.Adam(eps) on log_alpha (no amsgrad, no weight decay); alpha = exp(log_alpha).  Advances the round counter.
__global__ void k_dsac_entropy(int B, const float *__restrict__ ent, float target_entropy, float *__restrict__ log_alpha /* [4]: w m v - */,
                               float *__restrict__ alpha, AdamHp h, const DsacScal *__restrict__ scal, const int *__restrict__ round_idx,
                               const DsacCall *__restrict__ call, int autotune) {
    __shared__ float red[256];
    if (!autotune) {
        if (threadIdx.x == 0) *const_cast<int *>(round_idx) += 1;
        return;
    }
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) s += ent[b];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) {
        const float H = -(red[0] / (float)B), ea = expf(log_alpha[0]);
        const float g = ea * (H - target_entropy);        // the loss, and its derivative in log_alpha
        call->out_entropy[*round_idx] = g;
        const DsacScal sc = scal[*round_idx];
        float mm = log_alpha[1], vv = log_alpha[2], xx = 0.f;   // xx = max(0, v) = v: Adam without amsgrad
        const float p = adamw1(log_alpha[0], mm, vv, xx, g, h, sc.e_ss, sc.e_bc2s);
        log_alpha[0] = p; log_alpha[1] = mm; log_alpha[2] = vv;
        *alpha = expf(p);
        *const_cast<int *>(round_idx) += 1;
    }
}

}  // namespace

// ------------------------------------------------------------------ host side
struct prl_dsac {
    prl_dsac_cfg cfg;
    int Pa, Pc;                       // actor parameters; parameters of ONE critic
    int aW1, ab1, aW2, ab2, aW3, ab3;
    int cW1, cb1, cW2, cb2, cW3, cb3;
    float *actor, *actor_m, *actor_v, *actor_x;
    float *critic, *critic_m, *critic_v, *critic_x, *critic_t;
    float *log_alpha, *alpha;
    int64_t adam_step;
    // workspace
    float *S, *S2, *onehot, *R, *T, *h1, *h2, *logits, *dlogits, *ent, *P, *h1all, *c2all, *qall, *c1, *c2, *q, *dq, *dc2, *dc1,
        *dh2, *dh1, *y, *g_actor, *g_critic;
    int32_t *slots, *logical;
    DsacScal *scal;
    DsacCall *call;
    int *round_idx;
    bool use_graph;
    cudaGraphExec_t graph_exec;
    int graph_batch;
    const uint32_t *graph_buf;
    int launches_per_round;
    char *blk_host[2];
    cudaEvent_t blk_done[2];
    int blk_next;
    int64_t last_launches;
};

static int64_t al64(int64_t x) { return (x + 255) / 256 * 256; }

static void dsac_layout(prl_dsac *s) {
    const prl_dsac_cfg &c = s->cfg;
    int o = 0;
    s->aW1 = o; o += c.actor_h1 * c.obs_dim; s->ab1 = o; o += c.actor_h1;
    s->aW2 = o; o += c.actor_h2 * c.actor_h1; s->ab2 = o; o += c.actor_h2;
    s->aW3 = o; o += c.n_actions * c.actor_h2; s->ab3 = o; o += c.n_actions;
    s->Pa = o;
    const int D = c.obs_dim + c.n_actions;
    o = 0;
    s->cW1 = o; o += c.critic_h1 * D; s->cb1 = o; o += c.critic_h1;
    s->cW2 = o; o += c.critic_h2 * c.critic_h1; s->cb2 = o; o += c.critic_h2;
    s->cW3 = o; o += c.critic_h2; s->cb3 = o; o += 1;
    s->Pc = o;
}

static int dsac_check(const prl_dsac_cfg *c) {
    PRL_REQUIRE(c, "null cfg");
    PRL_REQUIRE(c->obs_dim > 0 && c->n_actions > 0 && c->actor_h1 > 0 && c->actor_h2 > 0 && c->critic_h1 > 0 && c->critic_h2 > 0,
                "dimensions must be positive");
    PRL_REQUIRE(c->max_batch > 0 && c->max_rounds > 0, "max_batch / max_rounds must be positive");
    return PRL_OK;
}

extern "C" int64_t prl_dsac_actor_param_count(const prl_dsac_cfg *c) {
    if (dsac_check(c)) return -1;
    prl_dsac t; t.cfg = *c; dsac_layout(&t);
    return t.Pa;
}
extern "C" int64_t prl_dsac_critic_param_count(const prl_dsac_cfg *c) {   // ONE critic; the twin vector holds two
    if (dsac_check(c)) return -1;
    prl_dsac t; t.cfg = *c; dsac_layout(&t);
    return t.Pc;
}

static size_t blk_bytes(const prl_dsac_cfg *c) { return (size_t)c->max_rounds * sizeof(DsacScal) + sizeof(DsacCall) + 16; }

struct DsacWs { int64_t off[40]; int64_t total; };
static DsacWs dsac_ws(const prl_dsac_cfg *c, int Pa, int Pc) {
    DsacWs w; int64_t o = 0; int k = 0;
    const int64_t B = c->max_batch, A = c->n_actions, O = c->obs_dim, BA = B * A;
    auto add = [&](int64_t floats) { w.off[k++] = o; o = al64(o + floats * 4); };
    add(B * O); add(B * O); add(B * A); add(B); add(B);                                   // S S2 onehot R T
    add(B * c->actor_h1); add(B * c->actor_h2); add(B * A); add(B * A); add(B);           // h1 h2 logits dlogits ent
    add(2 * B * c->critic_h1); add(2 * BA * c->critic_h1); add(2 * BA * c->critic_h2);   // P h1all c2all
    add(2 * BA);                                                                          // qall
    add(2 * B * c->critic_h1); add(2 * B * c->critic_h2); add(2 * B); add(2 * B);         // c1 c2 q dq
    add(2 * B * c->critic_h2); add(2 * B * c->critic_h1);                                 // dc2 dc1
    add(B * c->actor_h2); add(B * c->actor_h1); add(B);                                   // dh2 dh1 y
    add(Pa); add(2 * (int64_t)Pc);                                                        // g_actor g_critic
    add((int64_t)c->max_rounds * B); add((int64_t)c->max_rounds * B);                    // slots logical (int32)
    add((int64_t)(blk_bytes(c) + 3) / 4);                                                 // scal | call | round_idx
    w.total = o;
    return w;
}
extern "C" int64_t prl_dsac_workspace_bytes(const prl_dsac_cfg *c) {
    if (dsac_check(c)) return -1;
    prl_dsac t; t.cfg = *c; dsac_layout(&t);
    return dsac_ws(c, t.Pa, t.Pc).total;
}

extern "C" int prl_dsac_create(prl_dsac **out, const prl_dsac_cfg *cfg, float *actor_w, float *actor_m, float *actor_v, float *actor_vmax,
                               float *critic_w, float *critic_m, float *critic_v, float *critic_vmax, float *critic_target_w,
                               float *log_alpha4, float *alpha1, int64_t adam_step, void *workspace) {
    PRL_REQUIRE(out && actor_w && actor_m && actor_v && actor_vmax && critic_w && critic_m && critic_v && critic_vmax &&
                    critic_target_w && log_alpha4 && alpha1 && workspace, "null argument");
    int rc = dsac_check(cfg);
    if (rc) return rc;
    prl_dsac *s = new (std::nothrow) prl_dsac();
    if (!s) return fail(PRL_ENOMEM, "out of host memory");
    s->cfg = *cfg;
    dsac_layout(s);
    s->actor = actor_w; s->actor_m = actor_m; s->actor_v = actor_v; s->actor_x = actor_vmax;
    s->critic = critic_w; s->critic_m = critic_m; s->critic_v = critic_v; s->critic_x = critic_vmax; s->critic_t = critic_target_w;
    s->log_alpha = log_alpha4; s->alpha = alpha1;
    s->adam_step = adam_step;
    DsacWs w = dsac_ws(cfg, s->Pa, s->Pc);
    char *b = (char *)workspace;
    float **f[] = {&s->S, &s->S2, &s->onehot, &s->R, &s->T, &s->h1, &s->h2, &s->logits, &s->dlogits, &s->ent, &s->P, &s->h1all,
                   &s->c2all, &s->qall, &s->c1, &s->c2, &s->q, &s->dq, &s->dc2, &s->dc1, &s->dh2, &s->dh1, &s->y, &s->g_actor,
                   &s->g_critic};
    int k = 0;
    for (auto p : f) *p = (float *)(b + w.off[k++]);
    s->slots = (int32_t *)(b + w.off[k++]); s->logical = (int32_t *)(b + w.off[k++]);
    s->scal = (DsacScal *)(b + w.off[k++]);
    s->call = (DsacCall *)(s->scal + cfg->max_rounds); s->round_idx = (int *)(s->call + 1);
    s->blk_next = 0; s->use_graph = true; s->graph_exec = nullptr; s->graph_batch = 0; s->graph_buf = nullptr; s->last_launches = 0;
    static_assert(sizeof(DsacScal) % 8 == 0 && sizeof(DsacCall) % 8 == 0, "the call block follows the scalars 8-byte aligned");
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 2 && e == cudaSuccess; i++) {
        e = cudaHostAlloc((void **)&s->blk_host[i], blk_bytes(cfg), cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->blk_done[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { delete s; return fail(PRL_ECUDA, "prl_dsac_create: %s", cudaGetErrorString(e)); }
    *out = s;
    return PRL_OK;
}
extern "C" int prl_dsac_destroy(prl_dsac *s) {
    if (!s) return PRL_OK;
    for (int i = 0; i < 2; i++) { cudaEventSynchronize(s->blk_done[i]); cudaEventDestroy(s->blk_done[i]); cudaFreeHost(s->blk_host[i]); }
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    delete s;
    return PRL_OK;
}
extern "C" int64_t prl_dsac_adam_step(const prl_dsac *s) { return s ? s->adam_step : -1; }
extern "C" int prl_dsac_set_lr(prl_dsac *s, double actor_lr, double critic_lr) {
    PRL_REQUIRE(s, "null handle");
    PRL_REQUIRE(actor_lr >= 0.0 && critic_lr >= 0.0, "learning rates must be non-negative");
    s->cfg.actor_lr = actor_lr;
    s->cfg.critic_lr = critic_lr;
    return PRL_OK;
}

// one learner round, launched (or captured) on `st`; everything round-dependent is read on the device through
// s->scal / s->call / s->round_idx
static int dsac_round(prl_dsac *s, prl_buf *buf, int B, cudaStream_t st) {
    const prl_dsac_cfg &c = s->cfg;
    const int O = c.obs_dim, A = c.n_actions, D = O + A, BA = B * A;
    const int H1 = c.actor_h1, H2 = c.actor_h2, C1 = c.critic_h1, C2 = c.critic_h2;
    const long long Pc = s->Pc;
    // the decay and step sizes come from the per-round block; these carry the betas and eps only
    const AdamHp hw{1.f, (float)(1.0 - c.beta1), (float)c.beta2, (float)(1.0 - c.beta2), (float)c.eps};
    const AdamHp he{1.f, (float)(1.0 - c.beta1), (float)c.beta2, (float)(1.0 - c.beta2), (float)c.entropy_eps};
    GemmLauncher L; L.st = st;
    const float *aw = s->actor, *cw = s->critic, *ct = s->critic_t;
    const long long sC1 = (long long)B * C1, sC2 = (long long)B * C2, aC1 = (long long)BA * C1, aC2 = (long long)BA * C2;
    auto actor_forward = [&](const float *X) {
        L.fwd(mat(X, O), B, aw + s->aW1, O, 0, aw + s->ab1, 0, H1, O, true, s->h1, H1, 0);
        L.fwd(mat(s->h1, H1), B, aw + s->aW2, H1, 0, aw + s->ab2, 0, H2, H1, true, s->h2, H2, 0);
        L.fwd(mat(s->h2, H2), B, aw + s->aW3, H2, 0, aw + s->ab3, 0, A, H2, false, s->logits, A, 0);
    };
    const int eb = 256;
    int small = 0;
    auto critic_all_actions = [&](const float *net, const float *X) {   // qall[z][b * A + a], both critics (blockIdx.z)
        L.fwd(mat(X, O), B, net + s->cW1, D, Pc, nullptr, 0, C1, O, false, s->P, C1, sC1, 2);
        dim3 g((unsigned)((aC1 + eb - 1) / eb), 1, 2);
        k_dsac_expand<<<g, eb, 0, st>>>(B, A, C1, O, s->P, net + s->cW1, net + s->cb1, Pc, s->h1all);
        small++;
        L.fwd(mat(s->h1all, C1, aC1), BA, net + s->cW2, C1, Pc, net + s->cb2, Pc, C2, C1, true, s->c2all, C2, aC2, 2);
        L.fwd(mat(s->c2all, C2, aC2), BA, net + s->cW3, C2, Pc, net + s->cb3, Pc, 1, C2, false, s->qall, 1, BA, 2);
    };
    k_dsac_gather<<<(B * 32 + eb - 1) / eb, eb, 0, st>>>(buf->records, buf->lay, O, A, s->call, s->round_idx, B, s->S, s->S2, s->onehot,
                                                         s->R, s->T);
    small++;
    // ---------------- actor step (actor_critic_base.py:333-343; soft_actor_critic.py:247-286)
    actor_forward(s->S);
    critic_all_actions(cw, s->S);
    k_dsac_actor_loss<<<1, 256, 0, st>>>(B, A, s->logits, s->qall, s->alpha, s->dlogits, s->ent, s->call, s->round_idx);
    small++;
    {
        float *ga = s->g_actor;
        L.bwd_w(s->dlogits, A, 0, B, A, mat(s->h2, H2), H2, ga + s->aW3, H2, 0, ga + s->ab3, 0);
        L.bwd_x(s->dlogits, A, 0, B, A, aw + s->aW3, H2, 0, 0, H2, s->dh2, H2, 0, s->h2, H2, 0, false);
        L.bwd_w(s->dh2, H2, 0, B, H2, mat(s->h1, H1), H1, ga + s->aW2, H1, 0, ga + s->ab2, 0);
        L.bwd_x(s->dh2, H2, 0, B, H2, aw + s->aW2, H1, 0, 0, H1, s->dh1, H1, 0, s->h1, H1, 0, false);
        L.bwd_w(s->dh1, H1, 0, B, H1, mat(s->S, O), O, ga + s->aW1, O, 0, ga + s->ab1, 0);
        k_dsac_adamw<<<(s->Pa + eb - 1) / eb, eb, 0, st>>>(s->Pa, s->actor, s->actor_m, s->actor_v, s->actor_x, ga, hw, s->scal, 0,
                                                          s->round_idx, nullptr, 0.f, 0.f);
        small++;
    }
    // ---------------- critic step with the UPDATED actor (actor_critic_base.py:345-349; soft_actor_critic.py:180-245)
    actor_forward(s->S2);
    critic_all_actions(ct, s->S2);
    k_dsac_target<<<(B + 127) / 128, 128, 0, st>>>(B, A, s->logits, s->qall, s->alpha, (float)c.gamma, s->T, s->R, s->y);
    small++;
    L.fwd(mat2(s->S, O, O, s->onehot, A), B, cw + s->cW1, D, Pc, cw + s->cb1, Pc, C1, D, true, s->c1, C1, sC1, 2);
    L.fwd(mat(s->c1, C1, sC1), B, cw + s->cW2, C1, Pc, cw + s->cb2, Pc, C2, C1, true, s->c2, C2, sC2, 2);
    L.fwd(mat(s->c2, C2, sC2), B, cw + s->cW3, C2, Pc, cw + s->cb3, Pc, 1, C2, false, s->q, 1, B, 2);
    k_dsac_critic_loss<<<1, 256, 0, st>>>(B, s->q, s->y, s->dq, s->call, s->round_idx);
    small++;
    {
        float *gc = s->g_critic;
        L.bwd_w(s->dq, 1, B, B, 1, mat(s->c2, C2, sC2), C2, gc + s->cW3, C2, Pc, gc + s->cb3, Pc, 2);
        dim3 g2((B * C2 + eb - 1) / eb, 1, 2);
        k_head_bwd<<<g2, eb, 0, st>>>(B, C2, s->dq, cw + s->cW3, Pc, s->c2, s->dc2);
        small++;
        L.bwd_w(s->dc2, C2, sC2, B, C2, mat(s->c1, C1, sC1), C1, gc + s->cW2, C1, Pc, gc + s->cb2, Pc, 2);
        L.bwd_x(s->dc2, C2, sC2, B, C2, cw + s->cW2, C1, Pc, 0, C1, s->dc1, C1, sC1, s->c1, C1, sC1, false, 2);
        L.bwd_w(s->dc1, C1, sC1, B, C1, mat2(s->S, O, O, s->onehot, A), D, gc + s->cW1, D, Pc, gc + s->cb1, Pc, 2);
        const int n2p = 2 * s->Pc;
        k_dsac_adamw<<<(n2p + eb - 1) / eb, eb, 0, st>>>(n2p, s->critic, s->critic_m, s->critic_v, s->critic_x, gc, hw, s->scal, 1,
                                                        s->round_idx, s->critic_t, (float)c.tau, (float)(1.0 - c.tau));
        small++;
    }
    // ---------------- entropy coefficient (soft_actor_critic.py:151-178); also advances the round counter
    k_dsac_entropy<<<1, 256, 0, st>>>(B, s->ent, (float)c.target_entropy, s->log_alpha, s->alpha, he, s->scal, s->round_idx, s->call,
                                      c.autotune);
    small++;
    s->launches_per_round = L.count + small;
    return PRL_OK;
}

extern "C" int prl_dsac_learn(prl_dsac *s, prl_buf *buf, int rounds, int batch, float *out_actor_loss, float *out_critic_loss,
                              float *out_entropy_loss, int32_t *out_logical, void *stream_) {
    PRL_REQUIRE(s && buf && out_actor_loss && out_critic_loss && out_entropy_loss, "null argument");
    const prl_dsac_cfg &c = s->cfg;
    PRL_REQUIRE(rounds > 0 && rounds <= c.max_rounds && batch > 0 && batch <= c.max_batch, "rounds / batch outside the configured maxima");
    PRL_REQUIRE((buf->desc.flags & PRL_BUF_DISCRETE) && !(buf->desc.flags & PRL_BUF_CONTINUOUS),
                "discrete SAC needs a discrete-action buffer");
    PRL_REQUIRE(!(buf->desc.flags & PRL_BUF_DYNAMIC_ACTIONS),
                "discrete SAC needs a fixed action space: the buffer stores per-transition action sets, and the actor loss needs "
                "the current state's unavailable-action mask, which it does not store");
    PRL_REQUIRE(buf->shard_world <= 1, "discrete SAC does not learn from a sharded buffer");
    PRL_REQUIRE(buf->desc.obs_dim == c.obs_dim && buf->desc.n_actions == c.n_actions,
                "buffer dimensions (obs %d, %d actions) do not match the learner (obs %d, %d actions)", buf->desc.obs_dim,
                buf->desc.n_actions, c.obs_dim, c.n_actions);
    cudaStream_t st = (cudaStream_t)stream_;
    int rc = prl_buf_sample_indices(buf, rounds, batch, out_logical ? out_logical : s->logical, s->slots, stream_);
    if (rc) return rc;
    // per-call block: optimizer scalars of every round at the CURRENT learning rates (as torch evaluates them, in double)
    const int sb = s->blk_next; s->blk_next ^= 1;
    PRL_CUDA(cudaEventSynchronize(s->blk_done[sb]));
    DsacScal *hs = reinterpret_cast<DsacScal *>(s->blk_host[sb]);
    for (int r = 0; r < rounds; r++) {
        const double step = (double)(s->adam_step + r + 1);
        const double bc1 = 1.0 - pow(c.beta1, step), bc2s = sqrt(1.0 - pow(c.beta2, step));
        hs[r] = DsacScal{(float)(c.actor_lr / bc1), (float)bc2s, (float)(1.0 - c.actor_lr * c.weight_decay),
                         (float)(c.critic_lr / bc1), (float)bc2s, (float)(1.0 - c.critic_lr * c.weight_decay),
                         (float)(c.entropy_lr / bc1), (float)bc2s};
    }
    DsacCall *hc = reinterpret_cast<DsacCall *>(hs + c.max_rounds);
    hc->slots = s->slots; hc->out_actor = out_actor_loss; hc->out_critic = out_critic_loss; hc->out_entropy = out_entropy_loss;
    *reinterpret_cast<int *>(hc + 1) = 0;
    // scal | call | round_idx are contiguous on the device in the same order
    PRL_CUDA(cudaMemcpyAsync(s->scal, hs, (size_t)c.max_rounds * sizeof(DsacScal) + sizeof(DsacCall) + 4, cudaMemcpyHostToDevice, st));
    PRL_CUDA(cudaEventRecord(s->blk_done[sb], st));

    if (s->use_graph) {
        if (!s->graph_exec || s->graph_batch != batch || s->graph_buf != buf->records) {
            if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
            cudaStream_t cs;
            PRL_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t graph = nullptr;
            cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                dsac_round(s, buf, batch, cs);
                e = cudaStreamEndCapture(cs, &graph);
            }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&s->graph_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            cudaStreamDestroy(cs);
            if (e != cudaSuccess) { s->graph_exec = nullptr; return fail(PRL_ECUDA, "prl_dsac_learn: graph capture failed: %s", cudaGetErrorString(e)); }
            s->graph_batch = batch; s->graph_buf = buf->records;
        }
        for (int r = 0; r < rounds; r++) PRL_CUDA(cudaGraphLaunch(s->graph_exec, st));
    } else {
        for (int r = 0; r < rounds; r++) {
            rc = dsac_round(s, buf, batch, st);
            if (rc) return rc;
        }
    }
    PRL_CUDA(cudaGetLastError());
    s->adam_step += rounds;
    s->last_launches = (int64_t)s->launches_per_round * rounds;
    return PRL_OK;
}
extern "C" int prl_dsac_set_graph(prl_dsac *s, int enable) {
    PRL_REQUIRE(s, "null handle");
    s->use_graph = enable != 0;
    return PRL_OK;
}
extern "C" int64_t prl_dsac_last_launches(const prl_dsac *s) { return s ? s->last_launches : -1; }
