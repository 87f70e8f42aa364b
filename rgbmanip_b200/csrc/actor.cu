// Controller observation + actor forward of RGBManip's RL "global scheduling" policy (SURVEY 8(f)-2):
//   obs  = cat(pose_queue [T,N,7], bbox_queue [T,N,4]) permuted to [N, T*11] ++ one_hot(step - 1, T)      (rl_pose.py:173-187)
//   act  = Linear(60,96) ELU Linear(96,96) ELU Linear(96,32) ELU Linear(32,12)                              (module.py:24-34,89-91)
// One kernel: a block carries ACT_ENVS environments, the observation is assembled straight from the device-resident
// queues (float64 -> float32 like the reference's .float()), activations ping-pong in shared memory, weights are read
// through the read-only path (74 KB for the shipped sizes: L1/L2 resident).  fp32 throughout.
#include "stages.cuh"

namespace adp {

constexpr int ACT_ENVS = 8;
constexpr int ACT_THREADS = 256;
constexpr int ACT_MAXW = 256;       // widest layer

__global__ void __launch_bounds__(ACT_THREADS)
actor_forward_kernel(const ActorArgs a) {
    __shared__ float buf[2][ACT_ENVS][ACT_MAXW];
    const int e0 = blockIdx.x * ACT_ENVS, tid = threadIdx.x;
    const int in0 = a.dims[0], T = a.T;
    for (int i = tid; i < ACT_ENVS * in0; i += ACT_THREADS) {
        const int le = i / in0, c = i - le * in0, e = e0 + le;
        float v = 0.f;
        if (e < a.N) {
            if (c < T * 11) {
                const int t = c / 11, k = c - t * 11;
                v = k < 7 ? (float)a.pose[((size_t)t * a.N + e) * 7 + k] : (float)a.bbox[((size_t)t * a.N + e) * 4 + (k - 7)];
            } else {
                v = (c - T * 11 == a.step) ? 1.f : 0.f;
            }
            if (a.obs_out) a.obs_out[(size_t)e * in0 + c] = v;
        }
        buf[0][le][c] = v;
    }
    __syncthreads();
    int cur = 0;
    for (int l = 0; l < a.nlayers; ++l) {
        const int din = a.dims[l], dout = a.dims[l + 1];
        const bool last = l == a.nlayers - 1;
        for (int i = tid; i < ACT_ENVS * dout; i += ACT_THREADS) {
            const int le = i / dout, n = i - le * dout;
            const float* w = a.W[l] + (size_t)n * din;
            float acc = __ldg(a.b[l] + n);
            for (int k = 0; k < din; ++k) acc = fmaf(buf[cur][le][k], __ldg(w + k), acc);
            if (!last) {
                switch (a.activation) {
                    case 0: acc = acc > 0.f ? acc : expm1f(acc); break;                                   // nn.ELU(alpha = 1)
                    case 1: acc = 1.0507009873554804934193349852946f *
                                  (acc > 0.f ? acc : 1.6732632423543772848170429916717f * expm1f(acc)); break;   // nn.SELU
                    case 2: acc = fmaxf(acc, 0.f); break;                                                  // nn.ReLU
                    case 3: acc = acc > 0.f ? acc : 0.01f * acc; break;                                    // nn.LeakyReLU(0.01)
                    case 4: acc = tanhf(acc); break;
                    default: acc = 1.f / (1.f + expf(-acc)); break;                                        // nn.Sigmoid
                }
            }
            buf[cur ^ 1][le][n] = acc;
            if (last && e0 + le < a.N) a.act_out[(size_t)(e0 + le) * dout + n] = acc;
        }
        __syncthreads();
        cur ^= 1;
    }
}

int actor_forward(const ActorArgs& a, cudaStream_t stream) {
    ADP_CHECK_ARG(a.nlayers >= 1 && a.nlayers <= ACT_MAXL, "1..8 layers");
    ADP_CHECK_ARG(a.dims[0] == a.T * 12, "observation width must be T * 12");
    for (int l = 0; l <= a.nlayers; ++l) ADP_CHECK_ARG(a.dims[l] >= 1 && a.dims[l] <= ACT_MAXW, "layer width 1..256");
    ADP_CHECK_ARG(a.step >= -1 && a.step < a.T, "step index");
    ADP_CHECK_ARG(a.activation >= 0 && a.activation <= 5, "activation code");
    if (a.N == 0) return ADP_OK;
    actor_forward_kernel<<<cdiv(a.N, ACT_ENVS), ACT_THREADS, 0, stream>>>(a);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
