// verify_batch / verify_compressed_batch kernels (reference: verify, src/lib.rs:395-412; decompress_signature
// + decompress_point, src/lib.rs:260-268, 192-224).  The lane bodies are in lanes.cuh.
//
// One verification is a short pipeline of kernels, so that no kernel carries another phase's registers
// or instruction footprint:
//   (bjj_cuda.cu: k_decompress_prepare / k_batch_inverse / k_decompress_finish for compressed input) ->
//   k_verify_hash -> k_verify_split (EdDSA) -> k_verify_ec_vm || k_verify_exact
#include <stdlib.h>

#include "kernels.h"
#include "vmcurve.cuh"

using namespace bjj;

// resident CTAs per SM the compiler must make room for (register cap = 65536 / (128 * MINB)); the carry
// chains are dependent instruction streams, so the fma pipe needs >= 3-4 warps per SMSP to stay busy
#ifndef BJJ_VERIFY_HASH_MINB
#define BJJ_VERIFY_HASH_MINB 2
#endif
#define BJJ_VERIFY_EXACT_BLOCK 64
#ifndef BJJ_VERIFY_EXACT_REGS
#define BJJ_VERIFY_EXACT_REGS 240      // four 64-thread CTAs per SM
#endif

#if BJJ_VERIFY_HASH_MINB > 0
__global__ void __launch_bounds__(BJJ_BLOCK, BJJ_VERIFY_HASH_MINB) k_verify_hash(
#else
__global__ void __launch_bounds__(BJJ_BLOCK) k_verify_hash(
#endif
    size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax, const uint8_t* ay, const uint8_t* msg,
    const uint8_t* s_base, size_t s_stride, size_t s_off, const uint8_t* skip, uint8_t* hm, size_t plane, uint8_t* ok,
    int gate, ExactQueue qa, ExactQueue qr, uint32_t* gflags, int mode, int split, uint8_t* msg_status,
    unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    BJJ_CLAIM_LOOP(n, work)
    if (i < n)
    lane_verify_hash(r8x, r8y, ax, ay, msg, s_base, s_stride, s_off, skip, hm, plane, ok, i, gate != 0, qa, qr, flags, mode,
                     split != 0, msg_status);
    BJJ_FLAGS_END(gflags)
}

// half-size scalars (EdDSA lanes): pure integer-ALU work, small code, many resident warps
__global__ void __launch_bounds__(BJJ_BLOCK, 4) k_verify_split(size_t n, const uint8_t* s_base, size_t s_stride, size_t s_off,
                                                              uint8_t* hm, size_t plane, const uint8_t* ok) {
    BJJ_LANE_LOOP(n) lane_verify_split(s_base, s_stride, s_off, hm, plane, ok, i);
}

// ---- the Straus pass on shared-memory slots (vm.cuh / vmcurve.cuh) --------------------------------------------
// The algorithm and tables of verify_fast (lanes.cuh, the host-checkable statement of the same pass); every field
// operation is a call into ~20 KB of resident subroutines, a lane's working set is 11 slots (352 B) of shared
// memory, and BJJ_EC_VM_MINB CTAs (5 x 4 warps, 96 registers) share an SM.  Measured on one GPU against the inlined
// kernel of round 1 (228 registers, 2 CTAs per SM, 150 KB window body): 60.4 ms against 66.2 ms per 2^21 lanes,
// multiplier pipe 86 % against 66-78 % busy, `no_instruction` 0.17 against 1.2 stalls per issue
// (profiles/r2_ab_verify_ec.txt, profiles/r2_ncu_verify_ec_summary.txt).
#ifndef BJJ_EC_VM_MINB
#define BJJ_EC_VM_MINB 5
#endif
#define BJJ_EC_VM_SLOTS (BJJ_VM_REG_SLOTS + 2)
#ifndef BJJ_EC_PREFETCH
#define BJJ_EC_PREFETCH 1
#endif

__device__ __forceinline__ int vm_digit4(vm::Slot s, uint32_t top, int i) {      // signed radix-16 digit i in [0, 64]
    const uint32_t w = vm::ld_word(s, (i >> 3) & 7);
    return i == 64 ? (int)top : (int)((w >> ((i & 7) * 4)) & 15u) - 8;
}
__device__ __forceinline__ int vm_digit16(vm::Slot s, uint32_t top, int i) {     // signed radix-65536 digit i in [0, 16]
    const uint32_t w = vm::ld_word(s, (i >> 1) & 7);
    return i == 16 ? (int)top : (int)((w >> ((i & 1) * 16)) & 65535u) - 32768;
}

__device__ __forceinline__ void lane_verify_ec_vm(const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax, const uint8_t* ay,
                                                  const uint8_t* hm_in, size_t plane, uint8_t* ok, size_t i, const vm::Table& ta,
                                                  const vm::Table& tr, const CombEntry* comb, int mode) {
    using namespace vm;
    const Regs s = regs_at(0);
    const Slot su = slot(BJJ_VM_REG_SLOTS), sv = slot(BJJ_VM_REG_SLOTS + 1);
    uint32_t tops, vneg;
    int nwin;
    {
        uint32_t u[8], v[8];
        load_u256(u, hm_in, plane + i);
        load_u256(v, hm_in, 2 * plane + i);
        vneg = v[7] >> 31;
        v[7] &= 0x7FFFFFFFu;
        Recode4 ru, rv;
        recode4(ru, u);
        recode4(rv, v);
        nwin = recode4_windows(ru);
        const int nv = recode4_windows(rv);
        nwin = nwin > nv ? nwin : nv;
        nwin = __reduce_max_sync(__activemask(), nwin);      // one trip count per warp (leading digits of a narrower lane are 0)
        Fr t;
        fr_set(t, ru.w);
        st(su, t);
        fr_set(t, rv.w);
        st(sv, t);
        tops = ru.top | (rv.top << 1);
    }
    // tables of -sign(v) * 8A (pk itself for Schnorr) and of -R8
#pragma unroll 1
    for (int t = 0; t < 2; t++) {
        load_mont(s.X, t == 0 ? ax : r8x, i);
        load_mont(s.Y, t == 0 ? ay : r8y, i);
        from_affine(s);
        if (t == 0 && mode == BJJ_MODE_EDDSA) {
#pragma unroll 1
            for (int j = 0; j < 3; j++) dbl(s, j == 2);
        }
        if (t == 1 || !vneg) {       // negate: (-X, Y, Z, -T)
            neg(s.X, s.X);
            neg(s.T, s.T);
        }
        table_build(s, t == 0 ? ta : tr);
    }
    set_identity(s);
#pragma unroll 1
    for (int k = nwin - 1; k >= 0; k--) {
        // the two table entries of this window are requested into L2 before the doublings: the window tables (218 MB
        // per workspace) do not stay in L2, and a load is waited for at the next subroutine call
        const int da = vm_digit4(su, tops & 1u, k), dr = vm_digit4(sv, tops >> 1, k);
#if BJJ_EC_PREFETCH
        prefetch_l2(ta.entry(da < 0 ? -da : da));
        prefetch_l2(tr.entry(dr < 0 ? -dr : dr));
#endif
        if (k != nwin - 1) {
#pragma unroll 1
            for (int j = 0; j < 4; j++) dbl(s, j == 3);
        }
        add_digit(s, ta, da, true);
        add_digit(s, tr, dr, k == 0);       // T only where the B8 additions follow
    }
    // + w * B8: 16 signed 16-bit digits and the recoding carry against the fixed-base table, no doubling
    {
        uint32_t w[8];
        load_u256(w, hm_in, 3 * plane + i);
        Recode16 rw;
        recode16(rw, w);
        Fr t;
        fr_set(t, rw.w);
        st(su, t);
        tops = rw.top;
    }
#pragma unroll 1
    for (int k = BJJ_COMB_WINDOWS - 1; k >= 0; k--) add_comb(s, comb, k, vm_digit16(su, tops, k), k != 0);
    // acc == O = (0 : 1 : 1) ?   (Z != 0: complete formulas)
    Fr x, y, z;
    ld(x, s.X);
    ld(y, s.Y);
    ld(z, s.Z);
    ok[i] = (fr_is_zero(x) && fr_eq(y, z)) ? 1 : 0;
}

__global__ void __launch_bounds__(BJJ_VM_THREADS, BJJ_EC_VM_MINB) k_verify_ec_vm(size_t n, const uint8_t* r8x, const uint8_t* r8y,
                                                                               const uint8_t* ax, const uint8_t* ay, const uint8_t* hm,
                                                                               size_t plane, uint8_t* ok, U128* table,
                                                                               const CombEntry* comb, int mode, unsigned long long* work) {
    // two per-thread radix-16 tables (multiples of 8A and of R8), each thread's 2 x 9 entries contiguous
    const size_t tslot = 2 * ((size_t)blockIdx.x * blockDim.x + threadIdx.x);
    const vm::Table ta = vm::table_of(table, tslot), tr = vm::table_of(table, tslot + 1);
    BJJ_CLAIM_LOOP(n, work)
    if (i < n && ok[i] == BJJ_OK_PENDING) lane_verify_ec_vm(r8x, r8y, ax, ay, hm, plane, ok, i, ta, tr, comb, mode);
    fma_ballast(mode == BJJ_MODE_NEVER, (uint32_t)n, ok);      // never taken: see fr.cuh
}

// exact lanes: off-curve inputs replay the reference sequence (rare; fed by the queues of k_verify_hash).
// A warp claims 32 queue entries at a time from `work` -- first the "A off the curve" queue (the longer ladder), then the
// "only R8 off the curve" queue, so no warp ever mixes the two ladders -- until both are exhausted.
__global__ void __maxnreg__(BJJ_VERIFY_EXACT_REGS) k_verify_exact(const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s,
                                                                         const uint8_t* ax, const uint8_t* ay, const uint8_t* hm,
                                                                         uint8_t* ok, ExactQueue qa, ExactQueue qr,
                                                                         const CombEntry* comb, int mode, unsigned long long* work) {
    const uint32_t ca = *qa.count, cr = *qr.count, lane = threadIdx.x & 31;
    const unsigned long long ua = (ca + 31u) >> 5, total = ua + ((cr + 31u) >> 5);
    auto claim = [&]() -> unsigned long long {
        unsigned long long u = 0;
        if (lane == 0) u = atomicAdd(work, 1ull);
        return __shfl_sync(0xFFFFFFFFu, u, 0);
    };
    unsigned long long u = claim();
    // one loop per ladder (a unit that ends the first loop is the first of the second)
    for (; u < ua; u = claim()) {
        const uint32_t j = (uint32_t)u * 32 + lane;
        if (j < ca) lane_verify_exact<true>(r8x, r8y, s, ax, ay, hm, ok, qa.list[j], comb, mode);
    }
    for (; u < total; u = claim()) {
        const uint32_t j = (uint32_t)(u - ua) * 32 + lane;
        if (j < cr) lane_verify_exact<false>(r8x, r8y, s, ax, ay, hm, ok, qr.list[j], comb, mode);
    }
}

namespace bjjk {

int verify_hash_blocks_per_sm() { return blocks_per_sm(k_verify_hash); }
static const size_t kEcVmSmem = vm::slot_bytes(BJJ_EC_VM_SLOTS);
int verify_ec_blocks_per_sm() {
    static int per_sm = [] {
        cudaFuncSetAttribute((const void*)k_verify_ec_vm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEcVmSmem);
        cudaFuncSetAttribute((const void*)k_verify_ec_vm, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        int v = blocks_per_sm(k_verify_ec_vm, BJJ_VM_THREADS, kEcVmSmem);
        // BJJ_EC_CTAS_PER_SM=n (experiments): fewer resident CTAs than fit, e.g. to leave registers for the exact-lane kernel
        if (const char* e = getenv("BJJ_EC_CTAS_PER_SM")) {
            const int cap = atoi(e);
            if (cap >= 1 && cap < v) v = cap;
        }
        return v;
    }();
    return per_sm;
}

int verify_split_blocks_per_sm() { return blocks_per_sm(k_verify_split); }

void verify_hash(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax,
                 const uint8_t* ay, const uint8_t* msg, const uint8_t* s_base, size_t s_stride, size_t s_off,
                 const uint8_t* skip, uint8_t* hm, size_t plane, uint8_t* ok, bool gate, ExactQueue qa, ExactQueue qr,
                 uint32_t* gflags, int mode, bool split, uint8_t* msg_status, unsigned long long* work) {
    k_verify_hash<<<grid, BJJ_BLOCK, 0, st>>>(n, r8x, r8y, ax, ay, msg, s_base, s_stride, s_off, skip, hm, plane, ok, gate ? 1 : 0,
                                              qa, qr, gflags, mode, split ? 1 : 0, msg_status, work);
}
void verify_split(int grid, cudaStream_t st, size_t n, const uint8_t* s_base, size_t s_stride, size_t s_off, uint8_t* hm,
                  size_t plane, const uint8_t* ok) {
    k_verify_split<<<grid, BJJ_BLOCK, 0, st>>>(n, s_base, s_stride, s_off, hm, plane, ok);
}
void verify_ec(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax,
               const uint8_t* ay, const uint8_t* hm, size_t plane, uint8_t* ok, U128* table, const CombEntry* comb,
               int mode, unsigned long long* work) {
    k_verify_ec_vm<<<grid, BJJ_VM_THREADS, kEcVmSmem, st>>>(n, r8x, r8y, ax, ay, hm, plane, ok, table, comb, mode, work);
}
void verify_exact(int grid, cudaStream_t st, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s, const uint8_t* ax,
                  const uint8_t* ay, const uint8_t* hm, uint8_t* ok, ExactQueue qa, ExactQueue qr, const CombEntry* comb,
                  int mode, unsigned long long* work) {
    k_verify_exact<<<grid, BJJ_VERIFY_EXACT_BLOCK, 0, st>>>(r8x, r8y, s, ax, ay, hm, ok, qa, qr, comb, mode, work);
}

}  // namespace bjjk
