#include "msm_impl.cuh"
namespace porla {
PORLA_INSTANTIATE_CURVE(Bn254)

// curve-independent: the data-side FFT butterfly (msm.cu computes the Barrett constant and calls this)
void data_butterfly_launch(uint32_t* d_blocks, uint32_t n_blocks, uint32_t chunks, uint32_t m, const uint8_t* d_twiddles,
                           const uint32_t* lcm16, const uint32_t* mu17, cudaStream_t stream) {
    DataFftParams prm;
    for (int i = 0; i < 16; i++) prm.lcm[i] = lcm16[i];
    for (int i = 0; i < 17; i++) prm.mu[i] = mu17[i];
    data_butterfly_impl(d_blocks, n_blocks, chunks, m, d_twiddles, prm, stream);
}

// ---------------------------------------------------------------------------- KZG digest scalars (BN254 Fr)
// out[b] = sum_i f_(b,i) * p_i mod r: alpha * f_b(tau) of the client's trapdoor digest (compute_digest) when p_i = alpha
// tau^i.  The coefficients are reduced mod r and stay canonical; the powers are in Montgomery form, so the Montgomery
// product of the two is the canonical f_i p_i and the sum comes out canonical.  One block per record.
using Bn254Fr = Fp<Bn254FrParams>;
constexpr int kFrEvalThreads = 128;
__global__ void __launch_bounds__(kFrEvalThreads)
k_fr_poly_eval(const uint8_t* __restrict__ coeffs_be, const Bn254Fr* __restrict__ powers, uint32_t n, uint8_t* __restrict__ out) {
    __shared__ Bn254Fr sh[kFrEvalThreads];
    const uint32_t b = blockIdx.x;
    Bn254Fr acc = Bn254Fr::zero();
#pragma unroll 1
    for (uint32_t i = threadIdx.x; i < n; i += kFrEvalThreads) {
        Bn254Fr f;
        load_u256(coeffs_be, (size_t)b * n + i, 1, f.v);
        reduce_scalar<Bn254>(f.v);
        acc = acc + f * ld16(powers + i);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
#pragma unroll 1
    for (uint32_t o = kFrEvalThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] = sh[threadIdx.x] + sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) store_u256(out, b, 0, sh[0].v);
}

void fr_poly_eval_device(const uint8_t* d_coeffs_be, const void* d_powers, uint32_t n, uint32_t nbatch, uint8_t* d_out,
                         cudaStream_t stream) {
    device_init();
    if (!nbatch) return;
    k_fr_poly_eval<<<nbatch, kFrEvalThreads, 0, stream>>>(d_coeffs_be, reinterpret_cast<const Bn254Fr*>(d_powers), n, d_out);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}
}
