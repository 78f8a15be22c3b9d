// spsg_normals.cuh -- per-voxel normals of the sparse SDF (forward + gather backward).
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// per-voxel normals of the sparse SDF (producer of the raycaster's vals_normals)
// ---------------------------------------------------------------------------------------------

// loss.compute_normals_sparse (loss.py:285-306) = compute_normals_dense (:261-267) on the scattered volume + gather +
// per-chunk rotation + -normalize, as one gather kernel over the voxel index:
//   g   = central differences of the SDF at the voxel, absent neighbours count as 0 (the dense volume is zero-filled,
//         loss.py:288-289), g = 0 on the volume border (the -inf padding that is then zeroed, :293-296);
//   m   = R_chunk * g            (transform[b, :3, :3], :299-301; identity without a transform)
//   out = -m / max(|m|, 1e-5)    (F.normalize(p=2, eps=1e-5), :305)
struct NormalsArgs {
    const longlong4 *locs;
    const float *sdf;
    const float *transform;  // (B,4,4) row-major or NULL; (B*F,4,4) for the per-view kernels
    const int32_t *index;    // (B,Dz,Dy,Dx) voxel -> row, -1 = absent
    const float *grad_out;   // backward: dL/d out (N,3)
    float *out;              // forward: normals (N,3); backward pass 1: u = dL/dg (N,3)
    float *d_sdf;            // backward pass 2: (N,1)
    long long n;
    int dimx, dimy, dimz;
};

__device__ __forceinline__ float sdf_at(const NormalsArgs &a, size_t chunk_base, int x, int y, int z) {
    const int i = __ldg(a.index + chunk_base + ((size_t)z * a.dimy + y) * a.dimx + x);
    return i >= 0 ? __ldg(a.sdf + i) : 0.0f;
}

__device__ __forceinline__ bool normals_gradient(const NormalsArgs &a, const longlong4 l, float &gx, float &gy, float &gz) {
    const int z = (int)l.x, y = (int)l.y, x = (int)l.z;
    gx = gy = gz = 0.0f;
    if (x < 1 || y < 1 || z < 1 || x > a.dimx - 2 || y > a.dimy - 2 || z > a.dimz - 2) return false;  // border: zero
    const size_t base = (size_t)l.w * a.dimz * a.dimy * a.dimx;
    gx = sdf_at(a, base, x + 1, y, z) - sdf_at(a, base, x - 1, y, z);
    gy = sdf_at(a, base, x, y + 1, z) - sdf_at(a, base, x, y - 1, z);
    gz = sdf_at(a, base, x, y, z + 1) - sdf_at(a, base, x, y, z - 1);
    return true;
}

__device__ __forceinline__ void load_rotation(const NormalsArgs &a, long long chunk, float (&R)[9]) {
    if (a.transform) {
        const float *t = a.transform + chunk * 16;
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = 0; c < 3; c++) R[r * 3 + c] = __ldg(t + r * 4 + c);
    } else {
#pragma unroll
        for (int k = 0; k < 9; k++) R[k] = (k % 4 == 0) ? 1.0f : 0.0f;
    }
}

__global__ void __launch_bounds__(256) normals_forward_kernel(const NormalsArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const longlong4 l = a.locs[i];
    float gx, gy, gz, R[9];
    normals_gradient(a, l, gx, gy, gz);
    load_rotation(a, l.w, R);
    const float mx = R[0] * gx + R[1] * gy + R[2] * gz, my = R[3] * gx + R[4] * gy + R[5] * gz,
                mz = R[6] * gx + R[7] * gy + R[8] * gz;
    const float inv = 1.0f / fmaxf(sqrtf(mx * mx + my * my + mz * mz), 1e-5f);
    a.out[i * 3 + 0] = -(mx * inv);
    a.out[i * 3 + 1] = -(my * inv);
    a.out[i * 3 + 2] = -(mz * inv);
}

// backward pass 1: u = dL/dg per voxel (zero on the border), through -normalize and the rotation
__global__ void __launch_bounds__(256) normals_backward_u_kernel(const NormalsArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const longlong4 l = a.locs[i];
    float gx, gy, gz, R[9];
    float ux = 0.0f, uy = 0.0f, uz = 0.0f;
    if (normals_gradient(a, l, gx, gy, gz)) {
        load_rotation(a, l.w, R);
        const float mx = R[0] * gx + R[1] * gy + R[2] * gz, my = R[3] * gx + R[4] * gy + R[5] * gz,
                    mz = R[6] * gx + R[7] * gy + R[8] * gz;
        const float len = sqrtf(mx * mx + my * my + mz * mz);
        const float qx = __ldg(a.grad_out + i * 3 + 0), qy = __ldg(a.grad_out + i * 3 + 1), qz = __ldg(a.grad_out + i * 3 + 2);
        float dmx, dmy, dmz;  // dL/dm for out = -m / max(len, eps)
        if (len > 1e-5f) {
            const float inv = 1.0f / len;
            const float hx = mx * inv, hy = my * inv, hz = mz * inv, dot = hx * qx + hy * qy + hz * qz;
            dmx = -(qx - hx * dot) * inv; dmy = -(qy - hy * dot) * inv; dmz = -(qz - hz * dot) * inv;
        } else {
            dmx = -qx * 1e5f; dmy = -qy * 1e5f; dmz = -qz * 1e5f;
        }
        ux = R[0] * dmx + R[3] * dmy + R[6] * dmz;  // R^T
        uy = R[1] * dmx + R[4] * dmy + R[7] * dmz;
        uz = R[2] * dmx + R[5] * dmy + R[8] * dmz;
    }
    a.out[i * 3 + 0] = ux; a.out[i * 3 + 1] = uy; a.out[i * 3 + 2] = uz;
}

// Per-view normals (SPSG_FLAG_VIEW_NORMALS renders): g once per voxel, then out[(i*F + f)*3 ..] = -normalize(R_{b*F+f} g)
// with the arithmetic of normals_forward_kernel; transform is (B*F,4,4), one rotation per image.
__global__ void __launch_bounds__(256) normals_forward_views_kernel(const NormalsArgs a, int views) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const longlong4 l = a.locs[i];
    float gx, gy, gz, R[9];
    normals_gradient(a, l, gx, gy, gz);
    for (int f = 0; f < views; f++) {
        load_rotation(a, l.w * views + f, R);
        const float mx = R[0] * gx + R[1] * gy + R[2] * gz, my = R[3] * gx + R[4] * gy + R[5] * gz,
                    mz = R[6] * gx + R[7] * gy + R[8] * gz;
        const float inv = 1.0f / fmaxf(sqrtf(mx * mx + my * my + mz * mz), 1e-5f);
        float *o = a.out + ((size_t)i * views + f) * 3;
        o[0] = -(mx * inv);
        o[1] = -(my * inv);
        o[2] = -(mz * inv);
    }
}

// backward pass 1 of the per-view normals: u = sum over f, in view order, of view f's dL/dg (normals_backward_u_kernel's
// formula with grad_out row (i, f) and image b*F+f's rotation)
__global__ void __launch_bounds__(256) normals_backward_u_views_kernel(const NormalsArgs a, int views) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const longlong4 l = a.locs[i];
    float gx, gy, gz, R[9];
    float ux = 0.0f, uy = 0.0f, uz = 0.0f;
    if (normals_gradient(a, l, gx, gy, gz)) {
        for (int f = 0; f < views; f++) {
            load_rotation(a, l.w * views + f, R);
            const float mx = R[0] * gx + R[1] * gy + R[2] * gz, my = R[3] * gx + R[4] * gy + R[5] * gz,
                        mz = R[6] * gx + R[7] * gy + R[8] * gz;
            const float len = sqrtf(mx * mx + my * my + mz * mz);
            const float *q = a.grad_out + ((size_t)i * views + f) * 3;
            const float qx = __ldg(q + 0), qy = __ldg(q + 1), qz = __ldg(q + 2);
            float dmx, dmy, dmz;
            if (len > 1e-5f) {
                const float inv = 1.0f / len;
                const float hx = mx * inv, hy = my * inv, hz = mz * inv, dot = hx * qx + hy * qy + hz * qz;
                dmx = -(qx - hx * dot) * inv; dmy = -(qy - hy * dot) * inv; dmz = -(qz - hz * dot) * inv;
            } else {
                dmx = -qx * 1e5f; dmy = -qy * 1e5f; dmz = -qz * 1e5f;
            }
            const float vx = R[0] * dmx + R[3] * dmy + R[6] * dmz, vy = R[1] * dmx + R[4] * dmy + R[7] * dmz,
                        vz = R[2] * dmx + R[5] * dmy + R[8] * dmz;
            ux += vx; uy += vy; uz += vz;
        }
    }
    a.out[i * 3 + 0] = ux; a.out[i * 3 + 1] = uy; a.out[i * 3 + 2] = uz;
}

// backward pass 2: the SDF value of voxel j enters g of its six neighbours with weight +-1 -- a gather, no atomics
__global__ void __launch_bounds__(256) normals_backward_gather_kernel(const NormalsArgs a) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.n) return;
    const longlong4 l = a.locs[j];
    const int z = (int)l.x, y = (int)l.y, x = (int)l.z;
    const size_t base = (size_t)l.w * a.dimz * a.dimy * a.dimx;
    const float *u = a.out;
    auto at = [&](int xx, int yy, int zz, int comp) -> float {
        if (xx < 0 || yy < 0 || zz < 0 || xx >= a.dimx || yy >= a.dimy || zz >= a.dimz) return 0.0f;
        const int i = __ldg(a.index + base + ((size_t)zz * a.dimy + yy) * a.dimx + xx);
        return i >= 0 ? __ldg(u + (size_t)i * 3 + comp) : 0.0f;
    };
    a.d_sdf[j] = (at(x - 1, y, z, 0) - at(x + 1, y, z, 0)) + (at(x, y - 1, z, 1) - at(x, y + 1, z, 1)) +
                 (at(x, y, z - 1, 2) - at(x, y, z + 1, 2));
}
