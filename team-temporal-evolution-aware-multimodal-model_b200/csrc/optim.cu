// Multi-tensor optimizer step for the trainable head parameters (SURVEY 8f "next": fused AdamW; the learner builds
// torch.optim.AdamW / SGD over net.parameters(), models/proof.py:357-361, and steps it at :445).
// One launch updates every listed tensor: the pointer table travels by value, so the launch can be captured behind
// the backward (and its gradient exchange) in the same CUDA graph.  Element-wise, no reductions -> bit-reproducible.
#include "common.cuh"

namespace team {

constexpr int OPT_MAX_TENSORS = 48;
struct OptList {
    float* p[OPT_MAX_TENSORS];
    const float* g[OPT_MAX_TENSORS];
    float* m[OPT_MAX_TENSORS];
    float* v[OPT_MAX_TENSORS];
    long long blk0[OPT_MAX_TENSORS + 1];      // first block of tensor i (1024 elements per block)
    long long n[OPT_MAX_TENSORS];
    int count;
};

// torch.optim.AdamW (decoupled weight decay, bias-corrected, amsgrad=False, maximize=False):
//   p *= 1 - lr wd;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
__global__ void __launch_bounds__(256)
adamw_kernel(const __grid_constant__ OptList L, float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt,
             const long long* __restrict__ step_dev) {
    __shared__ float bc[2];
    pdl_trigger();
    pdl_wait();
    if (step_dev != nullptr) {          // graph form: the step count lives on the device (adamw_tick_kernel advances it)
        // one thread per CTA: two double-precision pow() in EVERY thread made this kernel 26 us instead of 8 (tools/timeline_train.py)
        if (threadIdx.x == 0) {
            const double t = (double)(*step_dev + 1);
            bc[0] = (float)(1.0 - pow((double)b1, t));
            bc[1] = (float)sqrt(1.0 - pow((double)b2, t));
        }
        __syncthreads();
        bc1 = bc[0];
        bc2_sqrt = bc[1];
    }
    int t = 0;
    for (int i = 1; i < L.count; ++i)
        if ((long long)blockIdx.x >= L.blk0[i]) t = i;
    const long long base = ((long long)blockIdx.x - L.blk0[t]) * 1024;
    const float step_size = lr / bc1;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const long long i = base + q * 256 + threadIdx.x;
        if (i >= L.n[t]) break;
        const float g = L.g[t][i];
        float p = L.p[t][i] * (1.0f - lr * wd);
        const float m = b1 * L.m[t][i] + (1.0f - b1) * g;
        const float v = b2 * L.v[t][i] + (1.0f - b2) * g * g;
        L.m[t][i] = m; L.v[t][i] = v;
        p -= step_size * (m / (sqrtf(v) / bc2_sqrt + eps));
        L.p[t][i] = p;
    }
}

// one launch instead of four device-to-device copies: a batch (image rows, text rows, state ids, labels) into the static input
// buffers of a captured step (train.TrainStep.load) - between two graph replays the host-side launch latency of the copies
// was 17 us of a 350 us step
__global__ void __launch_bounds__(256)
copy_batch_kernel(const float4* __restrict__ image, const float4* __restrict__ text, const int64_t* __restrict__ state,
                  const int64_t* __restrict__ labels, long long n4, long long batch, float4* __restrict__ d_image,
                  float4* __restrict__ d_text, int64_t* __restrict__ d_state, int64_t* __restrict__ d_labels) {
    pdl_trigger();
    pdl_wait();
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i < n4) { d_image[i] = image[i]; d_text[i] = text[i]; }
    if (i < batch) { d_state[i] = state[i]; d_labels[i] = labels[i]; }
}

__global__ void adamw_tick_kernel(long long* step_dev) {
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x == 0) *step_dev += 1;
}

}  // namespace team

using namespace team;

static int adamw_launch(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                        float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                        float weight_decay, int64_t step, long long* step_dev, void* stream);

extern "C" int team_adamw_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                               float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2,
                               float eps, float weight_decay, int64_t step, void* stream) {
    TEAM_REQUIRE(step >= 1, "adamw: step counts from 1");
    return adamw_launch(n_tensors, params, grads, exp_avg, exp_avg_sq, numel, lr, beta1, beta2, eps, weight_decay, step, nullptr, stream);
}

extern "C" int team_adamw_step_graph(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                                     float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2,
                                     float eps, float weight_decay, int64_t* step_dev, int32_t advance, void* stream) {
    TEAM_REQUIRE(step_dev != nullptr, "adamw: null step counter");
    int rc = adamw_launch(n_tensors, params, grads, exp_avg, exp_avg_sq, numel, lr, beta1, beta2, eps, weight_decay, 1,
                          reinterpret_cast<long long*>(step_dev), stream);
    if (rc) return rc;
    if (advance) TEAM_LAUNCH(adamw_tick_kernel, 1, 32, 0, (cudaStream_t)stream, reinterpret_cast<long long*>(step_dev));
    return TEAM_OK;
}

static int adamw_launch(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                        float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                        float weight_decay, int64_t step, long long* step_dev, void* stream) {
    TEAM_REQUIRE(n_tensors >= 0 && n_tensors <= OPT_MAX_TENSORS, "adamw: %d tensors (max %d per call)", n_tensors, OPT_MAX_TENSORS);
    TEAM_REQUIRE(n_tensors == 0 || (params && grads && exp_avg && exp_avg_sq && numel), "adamw: null table");
    if (n_tensors == 0) return TEAM_OK;
    OptList L;
    memset(&L, 0, sizeof(L));
    long long blocks = 0;
    for (int i = 0; i < n_tensors; ++i) {
        // a tensor without elements may have null pointers (torch gives an empty tensor none): no block maps to it
        TEAM_REQUIRE(numel[i] >= 0 && (numel[i] == 0 || (params[i] && grads[i] && exp_avg[i] && exp_avg_sq[i])), "adamw: bad tensor %d", i);
        L.p[i] = params[i]; L.g[i] = grads[i]; L.m[i] = exp_avg[i]; L.v[i] = exp_avg_sq[i]; L.n[i] = numel[i];
        L.blk0[i] = blocks;
        blocks += (numel[i] + 1023) / 1024;
    }
    L.blk0[n_tensors] = blocks;
    L.count = n_tensors;
    if (blocks == 0) return TEAM_OK;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    TEAM_LAUNCH(adamw_kernel, blocks, 256, 0, (cudaStream_t)stream, L, lr, beta1, beta2, eps, weight_decay, (float)bc1, (float)sqrt(bc2), (const long long*)step_dev);
    return TEAM_OK;
}

extern "C" int team_copy_batch(const float* image, const float* text, const int64_t* state_ids, const int64_t* labels, int64_t batch,
                               float* d_image, float* d_text, int64_t* d_state_ids, int64_t* d_labels, void* stream) {
    TEAM_REQUIRE(image && text && state_ids && labels && d_image && d_text && d_state_ids && d_labels && batch >= 1, "copy_batch: bad arguments");
    TEAM_REQUIRE(((reinterpret_cast<uintptr_t>(image) | reinterpret_cast<uintptr_t>(text) | reinterpret_cast<uintptr_t>(d_image) |
                   reinterpret_cast<uintptr_t>(d_text)) & 15) == 0, "copy_batch: feature rows must be 16-byte aligned");
    const long long n4 = (long long)batch * D / 4;
    TEAM_LAUNCH(copy_batch_kernel, (n4 + 255) / 256, 256, 0, (cudaStream_t)stream, reinterpret_cast<const float4*>(image),
                reinterpret_cast<const float4*>(text), state_ids, labels, n4, (long long)batch, reinterpret_cast<float4*>(d_image),
                reinterpret_cast<float4*>(d_text), d_state_ids, d_labels);
    return TEAM_OK;
}
