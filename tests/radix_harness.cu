// radix_harness.cu — test-only C ABI over the library's radix sort (microcket_b200/csrc/radix_sort.cuh), which the product's C ABI
// does not expose: tests/test_gpu_radix_edges.py compiles it into a temporary directory and checks the sort itself against a
// numpy stable lexsort.  Linked against libmicrocket_b200.so only for mk_set_error / mk_sm_count / mk_last_error.
//   build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -shared -I microcket_b200/csrc \
//               tests/radix_harness.cu -L microcket_b200 -lmicrocket_b200 -Xlinker -rpath=$PWD/microcket_b200 -o <tmp>/libradix_harness.so
// Every entry point sorts the device buffers in place on the default stream, synchronises, and reports what the device plan
// decided: out[0] = final_buf (the buffer that holds the result), out[1] = n_exec (passes that ran).  *launches counts the
// kernels radix_sort() enqueued (0 when it refused the call).  ws_n sizes the workspace (RadixWs::max_n).
#include <algorithm>
#include "mk_common.cuh"
#include "radix_sort.cuh"

static int rh_schedule(const int *bytes, int n_pass, int key_bytes, RadixSchedule *sch) {
    if (n_pass < 1 || n_pass > RS_MAX_PASSES) { mk_set_error("radix_harness: %d passes", n_pass); return MK_ERR_ARG; }
    sch->n_pass = n_pass;
    for (int p = 0; p < n_pass; ++p) {
        if (bytes[p] < 0 || bytes[p] >= key_bytes) { mk_set_error("radix_harness: byte %d", bytes[p]); return MK_ERR_ARG; }
        sch->byte_of[p] = bytes[p];
    }
    return MK_OK;
}

static int rh_finish(RadixWs &ws, u32 *out) {
    MK_CUDA(cudaDeviceSynchronize());
    MK_CUDA(cudaGetLastError());
    RadixPlan hp;
    MK_CUDA(cudaMemcpy(&hp, ws.plan.p, sizeof hp, cudaMemcpyDeviceToHost));
    out[0] = hp.final_buf; out[1] = hp.n_exec;
    return MK_OK;
}

extern "C" const char *rh_last_error(void) { return mk_last_error(); }

// KV64: u64 keys in k0 (k1 scratch), u32 values in v0 (v1 scratch); iota_vals = 1 makes the first executed pass write the input index
extern "C" int rh_sort_kv64(u64 *k0, u64 *k1, u32 *v0, u32 *v1, u64 n, const int *bytes, int n_pass, int iota_vals, size_t ws_n,
                            u32 *out, u64 *launches) {
    *launches = 0;
    RadixSchedule sch;
    MK_TRY(rh_schedule(bytes, n_pass, 8, &sch));
    RadixWs ws;
    MK_TRY(ws.alloc(ws_n));
    KV64::Bufs b; b.k[0] = k0; b.k[1] = k1; b.v[0] = v0; b.v[1] = v1;
    MK_TRY(radix_sort<KV64>(b, n, sch, ws, iota_vals, mk_sm_count(0), 0, launches));
    return rh_finish(ws, out);
}

// the histograms of every scheduled byte taken by a kernel of the caller, as k_pack_keys (pairs.cu) does: whole warps stay in the
// loop, lanes past the end pass valid = false
static __global__ void __launch_bounds__(256) k_rh_hist(const uint4 *k, u64 n, RadixSchedule sch, RadixPlan *plan) {
    extern __shared__ u32 s_hist[];
    for (int i = threadIdx.x; i < sch.n_pass * 256; i += 256) s_hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const u64 n_round = (n + 31) & ~(u64)31;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += (u64)gridDim.x * blockDim.x) {
        const bool valid = i < n;
        uint4 r = make_uint4(0, 0, 0, 0);
        if (valid) r = k[i];
        radix_hist_add<Rec16>(s_hist, sch, r, valid, lane);
    }
    __syncthreads();
    radix_hist_flush(s_hist, sch.n_pass, plan);
}

// Rec16: 16-byte records in k0 (k1 scratch) sorted on the scheduled bytes (0..15); hist_done = 1 takes the histograms with
// k_rh_hist first and lets radix_sort() skip its own
extern "C" int rh_sort_rec16(uint4 *k0, uint4 *k1, u64 n, const int *bytes, int n_pass, int hist_done, size_t ws_n, u32 *out, u64 *launches) {
    *launches = 0;
    RadixSchedule sch;
    MK_TRY(rh_schedule(bytes, n_pass, 16, &sch));
    RadixWs ws;
    MK_TRY(ws.alloc(ws_n));
    Rec16::Bufs b; b.k[0] = k0; b.k[1] = k1; b.v[0] = b.v[1] = nullptr;
    if (hist_done && n < (1ull << 30) && n <= ws.max_n) {
        const int sms = mk_sm_count(0);
        MK_CUDA(cudaMemsetAsync(ws.plan.p, 0, sizeof(RadixPlan), 0));
        const int grid = (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)sms * 8));
        k_rh_hist<<<grid, 256, sch.n_pass * 256 * 4, 0>>>(k0, n, sch, ws.plan.as<RadixPlan>());
        MK_CUDA(cudaGetLastError());
    }
    MK_TRY(radix_sort<Rec16>(b, n, sch, ws, 0, mk_sm_count(0), 0, launches, hist_done != 0));
    return rh_finish(ws, out);
}
