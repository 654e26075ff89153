// msm_batch kernels: R = sum_i k_i * P_i by bucket accumulation (lane bodies and the pipeline: msm.cuh).
#include <cub/device/device_radix_sort.cuh>

#include "kernels.h"
#include "msm.cuh"

using namespace bjj;

// every bucket to the identity (once per call: the chunks of a host call accumulate into the same buckets)
__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_clear(size_t nb, uint8_t* buckets) {
    BJJ_LANE_LOOP(nb) {
        PointExt id;
        ext_identity(id);
        msm_store_ext(buckets, i, id);
    }
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_prepare(size_t m, const uint8_t* px, const uint8_t* py, const uint8_t* k, MsmGeom g,
                                                           CombEntry* niels, uint32_t* keys, uint32_t* vals, uint8_t* status,
                                                           uint32_t* mflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(m) lane_msm_prepare(px, py, k, i, m, g, niels, keys, vals, status, flags);
    BJJ_FLAGS_END(mflags)
}

// level 1 over the sorted pairs, and the levels after it over the boundary lists; runs are claimed a warp at a time
__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_accumulate(size_t count, MsmPairs in, uint32_t nb, uint8_t* buckets,
                                                              uint32_t* out_keys, uint8_t* out_pts, unsigned long long* work) {
    const size_t runs = (count + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN;
    BJJ_CLAIM_LOOP(runs, work) if (i < runs) lane_msm_run(in, count, i, nb, buckets, out_keys, out_pts);
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_merge(size_t count, MsmPartials in, uint32_t nb, uint8_t* buckets,
                                                         uint32_t* out_keys, uint8_t* out_pts, unsigned long long* work) {
    const size_t runs = (count + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN;
    BJJ_CLAIM_LOOP(runs, work) if (i < runs) lane_msm_run(in, count, i, nb, buckets, out_keys, out_pts);
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_bucket_reduce(size_t segments, const uint8_t* buckets, MsmGeom g, uint8_t* seg_out) {
    BJJ_LANE_LOOP(segments) lane_msm_segment(buckets, g, i, seg_out);
}

// one CTA per window: W_w = the sum of the window's segment results (each thread a strided share, then a tree)
__global__ void __launch_bounds__(BJJ_BLOCK) k_msm_window_sum(const uint8_t* seg, MsmGeom g, uint8_t* wsum) {
    __shared__ PointExt part[BJJ_BLOCK];
    const uint32_t per_window = g.half / BJJ_MSM_SEG;
    const size_t base = (size_t)blockIdx.x * per_window;
    PointExt acc, p;
    ext_identity(acc);
    for (uint32_t t = threadIdx.x; t < per_window; t += blockDim.x) {
        msm_load_ext(p, seg, base + t);
        msm_add_ext(acc, acc, p);
    }
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int half = BJJ_BLOCK / 2; half > 0; half >>= 1) {
        if ((int)threadIdx.x < half) {
            msm_add_ext(acc, part[threadIdx.x], part[threadIdx.x + half]);
            part[threadIdx.x] = acc;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) msm_store_ext(wsum, blockIdx.x, part[0]);
}

// one thread: Horner over the windows, the result, and the call's flags into the context's word for bjj_sync
__global__ void __launch_bounds__(32) k_msm_finish(const uint8_t* wsum, MsmGeom g, const uint32_t* mflags, uint8_t* rx, uint8_t* ry,
                                                   uint32_t* gflags) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const uint32_t f = *mflags;
    lane_msm_finish(wsum, g, f, rx, ry);
    if (f) atomicOr(gflags, f);
}

namespace bjjk {

void msm_clear(int grid, cudaStream_t st, size_t nb, uint8_t* buckets) { k_msm_clear<<<grid, BJJ_BLOCK, 0, st>>>(nb, buckets); }
int msm_prepare_blocks_per_sm() { return blocks_per_sm(k_msm_prepare); }
void msm_prepare(int grid, cudaStream_t st, size_t m, const uint8_t* px, const uint8_t* py, const uint8_t* k, int bits,
                 CombEntry* niels, uint32_t* keys, uint32_t* vals, uint8_t* status, uint32_t* mflags) {
    k_msm_prepare<<<grid, BJJ_BLOCK, 0, st>>>(m, px, py, k, msm_geom(bits), niels, keys, vals, status, mflags);
}
size_t msm_sort_temp_bytes(size_t items, int key_bits) {
    size_t bytes = 0;
    cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int)items, 0, key_bits);
    return bytes;
}
cudaError_t msm_sort(cudaStream_t st, void* temp, size_t temp_bytes, uint32_t** keys, uint32_t** vals, size_t items, int key_bits) {
    cub::DoubleBuffer<uint32_t> k(keys[0], keys[1]), v(vals[0], vals[1]);
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, k, v, (int)items, 0, key_bits, st);
    if (k.Current() != keys[0]) std::swap(keys[0], keys[1]);
    if (v.Current() != vals[0]) std::swap(vals[0], vals[1]);
    return e;
}
int msm_accumulate_blocks_per_sm() { return blocks_per_sm(k_msm_accumulate); }
void msm_accumulate(int grid, cudaStream_t st, size_t count, const uint32_t* keys, const uint32_t* vals, const CombEntry* niels,
                    uint32_t nb, uint8_t* buckets, uint32_t* out_keys, uint8_t* out_pts, unsigned long long* work) {
    k_msm_accumulate<<<grid, BJJ_BLOCK, 0, st>>>(count, MsmPairs{keys, vals, niels}, nb, buckets, out_keys, out_pts, work);
}
int msm_merge_blocks_per_sm() { return blocks_per_sm(k_msm_merge); }
void msm_merge(int grid, cudaStream_t st, size_t count, const uint32_t* keys, const uint8_t* pts, uint32_t nb, uint8_t* buckets,
               uint32_t* out_keys, uint8_t* out_pts, unsigned long long* work) {
    k_msm_merge<<<grid, BJJ_BLOCK, 0, st>>>(count, MsmPartials{keys, pts}, nb, buckets, out_keys, out_pts, work);
}
int msm_bucket_reduce_blocks_per_sm() { return blocks_per_sm(k_msm_bucket_reduce); }
void msm_bucket_reduce(int grid, cudaStream_t st, int bits, const uint8_t* buckets, uint8_t* seg) {
    const MsmGeom g = msm_geom(bits);
    k_msm_bucket_reduce<<<grid, BJJ_BLOCK, 0, st>>>((size_t)g.windows * (g.half / BJJ_MSM_SEG), buckets, g, seg);
}
void msm_window_sum(cudaStream_t st, int bits, const uint8_t* seg, uint8_t* wsum) {
    const MsmGeom g = msm_geom(bits);
    k_msm_window_sum<<<g.windows, BJJ_BLOCK, 0, st>>>(seg, g, wsum);
}
void msm_finish(cudaStream_t st, int bits, const uint8_t* wsum, const uint32_t* mflags, uint8_t* rx, uint8_t* ry, uint32_t* gflags) {
    k_msm_finish<<<1, 32, 0, st>>>(wsum, msm_geom(bits), mflags, rx, ry, gflags);
}

}  // namespace bjjk
