// ppo.cu -- PPO dataset construction and loss as fused kernels.
//
// Replaces (reference, Python loops over lists of transition dicts):
//   pfrl/agents/ppo.py:36-53    _add_advantage_and_value_target_to_episode(s)
//                               (GAE: delta = r + g*nonterminal*V' - V,
//                                A = delta + g*l*A_next, v_teacher = A + V,
//                                reversed per episode segment)
//   pfrl/agents/ppo.py:476-478  torch.std_mean(all_advs, unbiased=False)
//   pfrl/agents/ppo.py:495      (advs - mean) / (std + 1e-8)
//   pfrl/agents/ppo.py:634-671  _lossfun (clipped surrogate, value loss with
//                               optional clipping, entropy bonus)
//
// Layout: rollout arrays are time-major [T, E] (E = environments), so the E
// threads of a scan read/write coalesced rows.  The recurrence is evaluated
// in fp64 (the reference's precision depends on the numpy version: float32
// or float64, SURVEY.md section 4) and stored as fp32.
#include <math.h>

#include "b2rl_internal.cuh"

namespace {

__device__ unsigned int g_gae_counter[B2RL_N_TICKETS]; // zero-initialised, self-resetting

struct GaeArgs {
    const float *reward, *nonterminal, *v, *v_next; // [T, E]
    const uint8_t *cut;   // [T, E] 1 = last transition of its episode segment
    const uint8_t *valid; // [T, E] 1 = slot holds a transition (or null = all)
    int T, E;
    double gamma, lambda;
    float *adv, *v_teacher; // [T, E]
    double *partial;        // [gridDim.x, 3] (count, sum, sumsq) scratch
    float *stats;           // [2] mean, std (unbiased=False) over valid entries
    unsigned ticket;        // completion counter of this launch
};

__global__ void __launch_bounds__(128) k_gae(GaeArgs a)
{
    __shared__ double sh[3][4];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    double cnt = 0.0, s1 = 0.0, s2 = 0.0;
    if (e < a.E) {
        double adv = 0.0;
        const double gl = a.gamma * a.lambda;
        for (int t = a.T - 1; t >= 0; t--) {
            const size_t i = (size_t)t * a.E + e;
            if (a.valid && !a.valid[i]) {
                adv = 0.0;
                continue;
            }
            if (a.cut[i]) adv = 0.0; // a new (later) segment starts after this one
            const double td = (double)a.reward[i] +
                              a.gamma * (double)a.nonterminal[i] * (double)a.v_next[i] -
                              (double)a.v[i];
            adv = td + gl * adv;
            const float advf = (float)adv;
            a.adv[i] = advf;
            a.v_teacher[i] = (float)(adv + (double)a.v[i]);
            cnt += 1.0;
            s1 += (double)advf;
            s2 += (double)advf * (double)advf;
        }
    }
    // block reduction of the moments
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        sh[0][warp] = cnt;
        sh[1][warp] = s1;
        sh[2][warp] = s2;
    }
    __syncthreads();
    __shared__ bool last;
    if (threadIdx.x == 0) {
        double c = 0, x = 0, y = 0;
        for (int w = 0; w < (blockDim.x >> 5); w++) {
            c += sh[0][w];
            x += sh[1][w];
            y += sh[2][w];
        }
        a.partial[blockIdx.x * 3 + 0] = c;
        a.partial[blockIdx.x * 3 + 1] = x;
        a.partial[blockIdx.x * 3 + 2] = y;
        __threadfence();
        const unsigned int prev = atomicInc(&g_gae_counter[a.ticket], gridDim.x - 1);
        last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        double c = 0, x = 0, y = 0;
        for (unsigned b = 0; b < gridDim.x; b++) {
            c += __ldcg(a.partial + b * 3 + 0);
            x += __ldcg(a.partial + b * 3 + 1);
            y += __ldcg(a.partial + b * 3 + 2);
        }
        const double mean = c > 0 ? x / c : 0.0;
        double var = c > 0 ? y / c - mean * mean : 0.0;
        if (var < 0) var = 0;
        a.stats[0] = (float)mean;
        a.stats[1] = (float)sqrt(var);
    }
}

// ---------------------------------------------------------------------------
// PPO loss: forward value + the three gradients in one pass.
// ---------------------------------------------------------------------------
__device__ unsigned int g_ppo_counter[B2RL_N_TICKETS];

struct PpoArgs {
    const float *log_prob, *entropy, *v_pred;              // [M] (require grad)
    const float *log_prob_old, *v_pred_old, *adv, *v_teacher; // [M]
    const float *adv_stats; // [2] mean, std or null (no standardisation)
    int M;
    float clip_eps, clip_eps_vf; // clip_eps_vf < 0: unclipped value loss
    float value_coef, entropy_coef;
    float *g_log_prob, *g_entropy, *g_v_pred; // [M] d loss / d input
    double *partial;  // [gridDim.x, 3]
    float *losses;    // [4] total, policy, value, entropy
    unsigned ticket;
};

__global__ void __launch_bounds__(256) k_ppo_loss(PpoArgs a)
{
    __shared__ double sh[3][8];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double lp = 0.0, lv = 0.0, le = 0.0;
    const float invM = 1.0f / (float)a.M;
    if (i < a.M) {
        float adv = a.adv[i];
        if (a.adv_stats) adv = (adv - a.adv_stats[0]) / (a.adv_stats[1] + 1e-8f); // ppo.py:495
        const float ratio = expf(a.log_prob[i] - a.log_prob_old[i]);
        const float s1 = ratio * adv;
        const float rc = fminf(fmaxf(ratio, 1.0f - a.clip_eps), 1.0f + a.clip_eps);
        const float s2 = rc * adv;
        lp = -(double)fminf(s1, s2);
        // d(-min(s1, s2))/d log_prob: s1 active (or tie inside the clip range)
        const bool inside = (ratio >= 1.0f - a.clip_eps) && (ratio <= 1.0f + a.clip_eps);
        float g = 0.f;
        if (s1 < s2 || (s1 == s2 && inside)) g = -adv * ratio;
        a.g_log_prob[i] = g * invM;

        const float v = a.v_pred[i], vt = a.v_teacher[i];
        const float d = v - vt;
        float lvi = d * d;
        float gv = 2.0f * d;
        if (a.clip_eps_vf >= 0.f) {
            const float vo = a.v_pred_old[i];
            const float lo = vo - a.clip_eps_vf, hi = vo + a.clip_eps_vf;
            const float vc = fminf(fmaxf(v, lo), hi);
            const float dc = vc - vt;
            const float lc = dc * dc;
            // d vc / dv of min(max(v, lo), hi) (ppo.py:28-33): autograd gives half the
            // gradient to each side of a max / min tie, so v == lo or v == hi passes 0.5
            const float pass = (v > lo ? 1.0f : v == lo ? 0.5f : 0.0f) *
                               (v < hi ? 1.0f : v == hi ? 0.5f : 0.0f);
            if (lc > lvi) {
                lvi = lc;
                gv = 2.0f * dc * pass;
            } else if (lc == lvi) {
                gv = 0.5f * (2.0f * d) + 0.5f * (2.0f * dc * pass);
            }
        }
        lv = (double)lvi;
        a.g_v_pred[i] = a.value_coef * gv * invM;
        le = -(double)a.entropy[i];
        a.g_entropy[i] = -a.entropy_coef * invM;
    }
    for (int o = 16; o > 0; o >>= 1) {
        lp += __shfl_xor_sync(0xffffffffu, lp, o);
        lv += __shfl_xor_sync(0xffffffffu, lv, o);
        le += __shfl_xor_sync(0xffffffffu, le, o);
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        sh[0][warp] = lp;
        sh[1][warp] = lv;
        sh[2][warp] = le;
    }
    __syncthreads();
    __shared__ bool last;
    if (threadIdx.x == 0) {
        double x = 0, y = 0, z = 0;
        for (int w = 0; w < (blockDim.x >> 5); w++) {
            x += sh[0][w];
            y += sh[1][w];
            z += sh[2][w];
        }
        a.partial[blockIdx.x * 3 + 0] = x;
        a.partial[blockIdx.x * 3 + 1] = y;
        a.partial[blockIdx.x * 3 + 2] = z;
        __threadfence();
        const unsigned int prev = atomicInc(&g_ppo_counter[a.ticket], gridDim.x - 1);
        last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        double x = 0, y = 0, z = 0;
        for (unsigned b = 0; b < gridDim.x; b++) {
            x += __ldcg(a.partial + b * 3 + 0);
            y += __ldcg(a.partial + b * 3 + 1);
            z += __ldcg(a.partial + b * 3 + 2);
        }
        const float policy = (float)(x / a.M), value = (float)(y / a.M),
                    ent = (float)(z / a.M);
        a.losses[1] = policy;
        a.losses[2] = value;
        a.losses[3] = ent;
        a.losses[0] = policy + a.value_coef * value + a.entropy_coef * ent; // ppo.py:665-669
    }
}

} // namespace

extern "C" int b2rl_gae(const float *reward, const float *nonterminal, const float *v,
                        const float *v_next, const uint8_t *cut, const uint8_t *valid, int32_t T,
                        int32_t E, double gamma, double lambda, float *adv, float *v_teacher,
                        double *scratch, float *stats, void *stream)
{
    B2RL_REQUIRE(reward && nonterminal && v && v_next && cut && adv && v_teacher && scratch &&
                     stats, B2RL_ERR_INVALID, "gae: null argument");
    B2RL_REQUIRE(T > 0 && E > 0, B2RL_ERR_RANGE, "gae: empty rollout");
    GaeArgs a{reward, nonterminal, v, v_next, cut, valid, T, E, gamma, lambda,
              adv, v_teacher, scratch, stats};
    a.ticket = b2rl_next_ticket();
    k_gae<<<(E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a);
    B2RL_CUDA(cudaGetLastError());
    return B2RL_OK;
}

extern "C" int b2rl_ppo_loss(const float *log_prob, const float *entropy, const float *v_pred,
                             const float *log_prob_old, const float *v_pred_old,
                             const float *adv, const float *v_teacher, const float *adv_stats,
                             int32_t M, float clip_eps, float clip_eps_vf, float value_coef,
                             float entropy_coef, float *g_log_prob, float *g_entropy,
                             float *g_v_pred, double *scratch, float *losses, void *stream)
{
    B2RL_REQUIRE(log_prob && entropy && v_pred && log_prob_old && adv && v_teacher &&
                     g_log_prob && g_entropy && g_v_pred && scratch && losses,
                 B2RL_ERR_INVALID, "ppo_loss: null argument");
    B2RL_REQUIRE(clip_eps_vf < 0.f || v_pred_old, B2RL_ERR_INVALID,
                 "ppo_loss: clipped value loss needs v_pred_old");
    B2RL_REQUIRE(M > 0, B2RL_ERR_RANGE, "ppo_loss: empty minibatch");
    PpoArgs a{log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher, adv_stats, M,
              clip_eps, clip_eps_vf, value_coef, entropy_coef, g_log_prob, g_entropy, g_v_pred,
              scratch, losses};
    a.ticket = b2rl_next_ticket();
    k_ppo_loss<<<(M + 255) / 256, 256, 0, (cudaStream_t)stream>>>(a);
    B2RL_CUDA(cudaGetLastError());
    return B2RL_OK;
}
