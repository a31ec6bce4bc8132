#include "msm_impl.cuh"
namespace porla {
PORLA_INSTANTIATE_CURVE(Secp256k1)

void table_import_jacobian_secp256k1(const uint32_t* d_xyz, const uint8_t* d_inf, uint32_t n, void* d_points_out,
                                     uint8_t* d_flags_out, PointTable* out, cudaStream_t stream) {
    device_init();
    using A = Affine<Secp256k1::F>;
    if (n) {
        k_import_jacobian<Secp256k1><<<(n + 127) / 128, 128, 0, stream>>>(d_xyz, d_inf, n, reinterpret_cast<A*>(d_points_out),
                                                                         d_flags_out);
        LAUNCHED();
        PORLA_CUDA(cudaGetLastError());
    }
    *out = PointTable{};
    out->d_points = d_points_out;
    out->d_flags = d_flags_out;
    out->n = n;
    out->curve = kCurveSecp256k1;
}
}
