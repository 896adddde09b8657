// xchg.cu — the multi-GPU exchange of packed pairs, written once: owner bucketing and the all-to-all in ONE kernel over
// NVLink peer memory (SURVEY.md §8e: "dedup reshuffles keys by hash of (chr1,chr2,pos1-bin) ... so each GPU owns a disjoint
// key range").
//
// Every rank owns a receive buffer (two halves, used by alternating epochs) and a control block; all ranks map all of them
// (cudaIpc handles between processes, plain peer pointers inside one process).  k_xchg_scatter walks the rank's pairs in
// tiles of 2048: owner = mix(chr1, chr2, pos1 / res) mod world (the same hash as mk_pairs_owner), the tile is regrouped by
// owner in shared memory, one system-scope atomicAdd per (tile, owner) reserves the slots in the OWNER's buffer, and the
// runs go out as coalesced 16-byte stores straight into the peer's HBM.  The last CTA publishes this rank's epoch in every
// peer's control block; k_xchg_wait on the consumer side spins until all ranks have published, then reads how many pairs
// arrived.  No count exchange, no host round trip before the data moves, no library collective on the data path.
// With res = the least common multiple of all binning resolutions (5 Mb for the default list, microcket:98) every
// duplicate AND every cell of every resolution has exactly one owner, so dedup and all COO counts need no further exchange.
#include <algorithm>
#include <cstdlib>
#include <vector>
#include "mk_common.cuh"

#define XC_MAX_WORLD 64
#define XC_T 256
#define XC_ITEMS 8
#define XC_TILE (XC_T * XC_ITEMS)

struct XchgCtrl {                        // lives in every rank's memory, written by its peers
    unsigned long long cursor[2];        // next free slot of receive half 0 / 1
    u32 overflow[2];                     // a peer could not place its pairs (capacity)
    u32 flag[XC_MAX_WORLD];              // flag[r] = last epoch rank r has completely delivered
    u32 blocks_done;                     // local: CTAs of the running scatter that have finished
    u32 pad[3];
};

struct XchgPeers { mk_pair *recv[XC_MAX_WORLD]; XchgCtrl *ctrl[XC_MAX_WORLD]; };

__host__ __device__ __forceinline__ u32 xc_owner_hash(u32 chr1, u32 chr2, u32 pbin) {     // == mk_owner_hash (pairs.cu)
    u32 h = (chr1 * 0x9E3779B1u) ^ (chr2 * 0x85EBCA77u) ^ (pbin * 0xC2B2AE3Du);
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}

__device__ __forceinline__ void st_release_sys_u32(u32 *p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys_u32(const u32 *p) { u32 v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

// part != NULL: the pairs are the `part[1]` records that END at index part[0] of `p` (both written on the device by the
// producer, e.g. one sam2pairs window), and nothing is published: several such launches make up one epoch, closed by
// k_xchg_publish.  part == NULL: p[0, n) is the rank's whole contribution and the last CTA publishes the epoch itself.
//
// Who owns a 16-byte record is a policy: the packed pairs' owner (above), the owner of a SAM-space krmdup key record
// {key, ord} (mix(key, tag) mod world; the sender stamps its rank into ord on the way out), or the rank named in such a
// record's ord (the way back to the record's origin).
struct XcOwnPair {
    static __device__ __forceinline__ u32 owner(const uint4 &r, u32 world, u32 res) { return xc_owner_hash(r.z & 0xFFFFu, r.z >> 16, r.x / res) % world; }
    static __device__ __forceinline__ uint4 out(const uint4 &r, u32) { return r; }
};
struct XcOwnKey {                        // ord = tag << 63 | rank << 40 | line (s2p.cu, mk_s2p_rmdup_*)
    static __device__ __forceinline__ u32 owner(const uint4 &r, u32 world, u32) {
        u64 k = ((u64)r.y << 32 | r.x) ^ ((u64)(r.w >> 31) * 0x9E3779B97F4A7C15ull);
        k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
        return (u32)(k % world);
    }
    static __device__ __forceinline__ uint4 out(uint4 r, u32 rank) { r.w |= rank << 8; return r; }
};
struct XcOwnRank {
    static __device__ __forceinline__ u32 owner(const uint4 &r, u32 world, u32) { return ((r.w >> 8) & (XC_MAX_WORLD - 1)) % world; }
    static __device__ __forceinline__ uint4 out(const uint4 &r, u32) { return r; }
};

template <class Own>
__global__ void __launch_bounds__(XC_T) k_xchg_scatter(const mk_pair *p, u64 n, const unsigned long long *part, XchgPeers peers, XchgCtrl *mine,
                                                        u32 world, u32 rank, u32 res, u32 epoch, u64 half_cap) {
    __shared__ uint4 s_pair[XC_TILE];
    __shared__ u32 s_cnt[XC_MAX_WORLD], s_off[XC_MAX_WORLD + 1], s_fill[XC_MAX_WORLD];
    __shared__ unsigned long long s_base[XC_MAX_WORLD];
    __shared__ u32 s_last;
    const u32 tid = threadIdx.x, half = epoch & 1u;
    if (part) { n = part[1]; p += part[0] - n; }
    const u64 n_tiles = (n + XC_TILE - 1) / XC_TILE;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (tid < XC_MAX_WORLD) { s_cnt[tid] = 0; s_fill[tid] = 0; }
        __syncthreads();
        uint4 r[XC_ITEMS]; u32 d[XC_ITEMS];
#pragma unroll
        for (int k = 0; k < XC_ITEMS; ++k) {
            const u64 i = tile * XC_TILE + (u64)k * XC_T + tid;
            d[k] = 0xFFFFFFFFu;
            if (i < n) {
                r[k] = ((const uint4 *)p)[i];
                d[k] = Own::owner(r[k], world, res);
                r[k] = Own::out(r[k], rank);
                atomicAdd(&s_cnt[d[k]], 1u);
            }
        }
        __syncthreads();
        if (tid == 0) { u32 run = 0; for (u32 w = 0; w < world; ++w) { s_off[w] = run; run += s_cnt[w]; } s_off[world] = run; }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < XC_ITEMS; ++k) if (d[k] != 0xFFFFFFFFu) s_pair[s_off[d[k]] + atomicAdd(&s_fill[d[k]], 1u)] = r[k];
        // one reservation per (tile, owner) in the owner's memory
        if (tid < world && s_cnt[tid]) s_base[tid] = atomicAdd_system(&peers.ctrl[tid]->cursor[half], (unsigned long long)s_cnt[tid]);
        __syncthreads();
        const u32 total = s_off[world];
        for (u32 j = tid; j < total; j += XC_T) {
            u32 w = 0;                                                   // owner of slot j: the run that contains it
            { u32 lo = 0, hi = world; while (hi - lo > 1) { const u32 m = (lo + hi) >> 1; if (s_off[m] <= j) lo = m; else hi = m; } w = lo; }
            const unsigned long long slot = s_base[w] + (j - s_off[w]);
            if (slot < half_cap) peers.recv[w][(u64)half * half_cap + slot] = *(const mk_pair *)&s_pair[j];
            else peers.ctrl[w]->overflow[half] = 1u;
        }
        __syncthreads();
    }
    if (part) { __threadfence_system(); return; }
    // ---- completion: the last CTA tells every peer that this rank's pairs of this epoch are all in place
    __threadfence_system();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&mine->blocks_done, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (s_last) {
        if (tid == 0) {
            mine->blocks_done = 0;
            // the half of the NEXT epoch was consumed before this kernel started (stream order) and no peer writes into it
            // before it has seen this epoch's flag: reset its cursor here
            mine->cursor[half ^ 1u] = 0; mine->overflow[half ^ 1u] = 0;
        }
        __threadfence_system();
        __syncthreads();
        if (tid < world) st_release_sys_u32(&peers.ctrl[tid]->flag[rank], epoch);
    }
}

// closes an epoch made of partial scatters (all of them earlier in the same stream): what the last CTA of a whole scatter does
__global__ void k_xchg_publish(XchgPeers peers, XchgCtrl *mine, u32 world, u32 rank, u32 epoch) {
    const u32 tid = threadIdx.x, half = epoch & 1u;
    if (tid == 0) { mine->cursor[half ^ 1u] = 0; mine->overflow[half ^ 1u] = 0; }
    __threadfence_system();
    __syncthreads();
    if (tid < world) st_release_sys_u32(&peers.ctrl[tid]->flag[rank], epoch);
}

// wait until every rank has delivered `epoch`, then publish the count.  A rank may already have published the next epoch
// (one host thread driving several ranks of a two-step exchange, mk_s2p_rmdup_decide): it only does so after it has waited
// for this epoch itself, so a flag at or past `epoch` means this epoch's data is in place.
// (bounded: a peer that died or failed never publishes; after `timeout_ns` the wait gives up and reports which rank is missing
// instead of hanging the GPU)
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__global__ void k_xchg_wait(XchgCtrl *mine, u32 world, u32 epoch, unsigned long long timeout_ns,
                            unsigned long long *out /* [0] pairs received, [1] overflow, [2] 1 + first rank that did not deliver */) {
    const u32 tid = threadIdx.x;
    if (tid == 0) out[2] = 0;
    __syncthreads();
    if (tid < world) {
        const unsigned long long t0 = global_ns();
        while ((int)(ld_acquire_sys_u32(&mine->flag[tid]) - epoch) < 0) {
            __nanosleep(200);
            if (global_ns() - t0 > timeout_ns) { atomicMax(&out[2], (unsigned long long)tid + 1ull); break; }
        }
    }
    __syncthreads();
    if (tid == 0) { out[0] = mine->cursor[epoch & 1u]; out[1] = mine->overflow[epoch & 1u]; }
}

struct mk_xchg {
    int device = 0, world = 1, rank = 0, sms = 148;
    size_t half_cap = 0;                  // pairs per receive half
    DevBuf recv, ctrl, out;
    XchgPeers peers;
    std::vector<void *> opened;           // IPC mappings to close
    bool connected = false;
    u32 epoch = 0;
    u64 launches = 0;
};

extern "C" int mk_xchg_create(int device, int world, int rank, size_t cap_pairs, mk_xchg **out) {
    if (!out || world < 1 || world > XC_MAX_WORLD || rank < 0 || rank >= world || cap_pairs == 0) { mk_set_error("mk_xchg_create: bad argument"); return MK_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(device));
    mk_xchg *x = new mk_xchg();
    x->device = device; x->world = world; x->rank = rank; x->sms = mk_sm_count(device); x->half_cap = cap_pairs;
    int rc = x->recv.alloc(2 * cap_pairs * sizeof(mk_pair));
    if (rc == MK_OK) rc = x->ctrl.alloc(sizeof(XchgCtrl));
    if (rc == MK_OK) rc = x->out.alloc(32);
    if (rc != MK_OK) { delete x; return rc; }
    if (cudaMemset(x->ctrl.p, 0, sizeof(XchgCtrl)) != cudaSuccess) { delete x; mk_set_error("mk_xchg_create: memset failed"); return MK_ERR_CUDA; }
    memset(&x->peers, 0, sizeof x->peers);
    x->peers.recv[rank] = x->recv.as<mk_pair>(); x->peers.ctrl[rank] = x->ctrl.as<XchgCtrl>();
    x->connected = world == 1;
    *out = x;
    return MK_OK;
}

extern "C" void mk_xchg_destroy(mk_xchg *x) {
    if (!x) return;
    cudaSetDevice(x->device);
    for (void *p : x->opened) cudaIpcCloseMemHandle(p);
    delete x;
}

// 128 bytes: the IPC handles of the receive buffer and of the control block (for ranks in OTHER processes)
extern "C" int mk_xchg_handle(mk_xchg *x, void *handle128) {
    if (!x || !handle128) { mk_set_error("mk_xchg_handle: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(x->device));
    cudaIpcMemHandle_t h[2];
    MK_CUDA(cudaIpcGetMemHandle(&h[0], x->recv.p));
    MK_CUDA(cudaIpcGetMemHandle(&h[1], x->ctrl.p));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle128, h, 128);
    return MK_OK;
}

// all_handles: world x 128 bytes in rank order (an all-gather of mk_xchg_handle, by any bootstrap the caller has)
extern "C" int mk_xchg_connect(mk_xchg *x, const void *all_handles) {
    if (!x || !all_handles) { mk_set_error("mk_xchg_connect: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(x->device));
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) continue;
        cudaIpcMemHandle_t h[2];
        memcpy(h, (const char *)all_handles + (size_t)r * 128, 128);
        void *pr = nullptr, *pc = nullptr;
        MK_CUDA(cudaIpcOpenMemHandle(&pr, h[0], cudaIpcMemLazyEnablePeerAccess));
        x->opened.push_back(pr);
        MK_CUDA(cudaIpcOpenMemHandle(&pc, h[1], cudaIpcMemLazyEnablePeerAccess));
        x->opened.push_back(pc);
        x->peers.recv[r] = (mk_pair *)pr; x->peers.ctrl[r] = (XchgCtrl *)pc;
    }
    x->connected = true;
    return MK_OK;
}

// ranks that live in ONE process (one context per GPU, or several on one GPU in the tests): plain pointers
extern "C" int mk_xchg_connect_local(mk_xchg *const *all, int world) {
    if (!all || world < 1 || world > XC_MAX_WORLD) { mk_set_error("mk_xchg_connect_local: bad argument"); return MK_ERR_ARG; }
    for (int a = 0; a < world; ++a) {
        if (!all[a] || all[a]->world != world || all[a]->rank != a) { mk_set_error("mk_xchg_connect_local: contexts must be given in rank order"); return MK_ERR_ARG; }
        MK_CUDA(cudaSetDevice(all[a]->device));
        for (int b = 0; b < world; ++b) {
            if (all[b]->device != all[a]->device) {
                int can = 0;
                MK_CUDA(cudaDeviceCanAccessPeer(&can, all[a]->device, all[b]->device));
                if (!can) { mk_set_error("mk_xchg_connect_local: device %d cannot access device %d", all[a]->device, all[b]->device); return MK_ERR_CUDA; }
                cudaError_t e = cudaDeviceEnablePeerAccess(all[b]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { mk_set_error("cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); return MK_ERR_CUDA; }
                cudaGetLastError();
            }
            all[a]->peers.recv[b] = all[b]->recv.as<mk_pair>(); all[a]->peers.ctrl[b] = all[b]->ctrl.as<XchgCtrl>();
        }
        all[a]->connected = true;
    }
    return MK_OK;
}

// Enqueue this rank's half of the exchange: its n pairs go to their owners.  Returns at once (no synchronisation).
extern "C" int mk_xchg_scatter_device(mk_xchg *x, const mk_pair *d_pairs, size_t n, uint32_t res, void *stream) {
    if (!x || res == 0 || (n && !d_pairs)) { mk_set_error("mk_xchg_scatter_device: bad argument"); return MK_ERR_ARG; }
    if (!x->connected) { mk_set_error("mk_xchg_scatter_device: mk_xchg_connect first"); return MK_ERR_STATE; }
    MK_CUDA(cudaSetDevice(x->device));
    x->epoch += 1;
    const u64 n_tiles = (n + XC_TILE - 1) / XC_TILE;
    const int grid = (int)std::max<u64>(1, std::min<u64>(n_tiles, (u64)x->sms * 4));
    k_xchg_scatter<XcOwnPair><<<grid, XC_T, 0, (cudaStream_t)stream>>>(d_pairs, n, nullptr, x->peers, x->ctrl.as<XchgCtrl>(), (u32)x->world, (u32)x->rank, res, x->epoch, x->half_cap);
    x->launches += 1;
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}

// The same exchange in pieces, so that it overlaps with the producer: begin an epoch, scatter any number of parts (each the
// d_part[1] pairs that end at index d_part[0] of d_base; both values live on the DEVICE, written by the producer, e.g. one
// sam2pairs window), then end the epoch.  All calls of one epoch go to ONE stream.
extern "C" int mk_xchg_begin(mk_xchg *x) {
    if (!x) { mk_set_error("mk_xchg_begin: null"); return MK_ERR_ARG; }
    if (!x->connected) { mk_set_error("mk_xchg_begin: mk_xchg_connect first"); return MK_ERR_STATE; }
    x->epoch += 1;
    return MK_OK;
}
extern "C" int mk_xchg_scatter_part_device(mk_xchg *x, const mk_pair *d_base, const uint64_t *d_part, uint32_t res, void *stream) {
    if (!x || !d_base || !d_part || res == 0 || x->epoch == 0) { mk_set_error("mk_xchg_scatter_part_device: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(x->device));
    k_xchg_scatter<XcOwnPair><<<x->sms * 2, XC_T, 0, (cudaStream_t)stream>>>(d_base, 0, (const unsigned long long *)d_part, x->peers, x->ctrl.as<XchgCtrl>(),
                                                                  (u32)x->world, (u32)x->rank, res, x->epoch, x->half_cap);
    x->launches += 1;
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}
extern "C" int mk_xchg_end_device(mk_xchg *x, void *stream) {
    if (!x || x->epoch == 0) { mk_set_error("mk_xchg_end_device: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(x->device));
    k_xchg_publish<<<1, XC_MAX_WORLD, 0, (cudaStream_t)stream>>>(x->peers, x->ctrl.as<XchgCtrl>(), (u32)x->world, (u32)x->rank, x->epoch);
    x->launches += 1;
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}

// Wait (on the device) until every rank's pairs of the current epoch have arrived; *d_recv points at them (inside this
// object's receive buffer, valid until the scatter after next), *n_recv is their number.  One host synchronisation.
extern "C" int mk_xchg_finish_device(mk_xchg *x, mk_pair **d_recv, size_t *n_recv, void *stream) {
    if (!x || !d_recv || !n_recv) { mk_set_error("mk_xchg_finish_device: bad argument"); return MK_ERR_ARG; }
    if (x->epoch == 0) { mk_set_error("mk_xchg_finish_device: no scatter has been enqueued"); return MK_ERR_STATE; }
    MK_CUDA(cudaSetDevice(x->device));
    cudaStream_t s = (cudaStream_t)stream;
    const char *to = getenv("MICROCKET_XCHG_TIMEOUT_S");
    const unsigned long long timeout_ns = (unsigned long long)(to ? atof(to) : 60.0) * 1000000000ull;
    k_xchg_wait<<<1, XC_MAX_WORLD, 0, s>>>(x->ctrl.as<XchgCtrl>(), (u32)x->world, x->epoch, timeout_ns, x->out.as<unsigned long long>());
    x->launches += 1;
    unsigned long long h[3] = {0, 0, 0};
    MK_CUDA(cudaMemcpyAsync(h, x->out.p, 24, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (h[2]) { mk_set_error("mk_xchg_finish_device: rank %llu did not deliver epoch %u within the timeout", h[2] - 1, x->epoch); return MK_ERR_STATE; }
    *d_recv = x->recv.as<mk_pair>() + (size_t)(x->epoch & 1u) * x->half_cap;
    *n_recv = (size_t)std::min<unsigned long long>(h[0], x->half_cap);
    if (h[1] || h[0] > x->half_cap) { mk_set_error("mk_xchg_finish_device: rank %d was sent %llu pairs, capacity %zu", x->rank, h[0], x->half_cap); return MK_ERR_CAPACITY; }
    return MK_OK;
}

// 16-byte records of the multi-rank SAM-space krmdup (s2p.cu): owner 1 = the key's owner, 2 = the rank in the record's
// ord.  d_part == NULL: the n records at d_rec are the rank's whole contribution to a new epoch, published at the end;
// else one part of the epoch opened by mk_xchg_begin, as mk_xchg_scatter_part_device.
int xchg_scatter_records(mk_xchg *x, const void *d_rec, u64 n, const unsigned long long *d_part, int owner, cudaStream_t s) {
    if (!x || (owner != 1 && owner != 2)) { mk_set_error("xchg_scatter_records: bad argument"); return MK_ERR_ARG; }
    if (!x->connected) { mk_set_error("xchg_scatter_records: mk_xchg_connect first"); return MK_ERR_STATE; }
    MK_CUDA(cudaSetDevice(x->device));
    if (!d_part) x->epoch += 1;
    else if (x->epoch == 0) { mk_set_error("xchg_scatter_records: mk_xchg_begin first"); return MK_ERR_STATE; }
    const u64 n_tiles = (n + XC_TILE - 1) / XC_TILE;
    const int grid = d_part ? x->sms * 2 : (int)std::max<u64>(1, std::min<u64>(n_tiles, (u64)x->sms * 4));
    auto k = owner == 1 ? k_xchg_scatter<XcOwnKey> : k_xchg_scatter<XcOwnRank>;
    k<<<grid, XC_T, 0, s>>>((const mk_pair *)d_rec, n, d_part, x->peers, x->ctrl.as<XchgCtrl>(), (u32)x->world, (u32)x->rank, 1u, x->epoch, x->half_cap);
    x->launches += 1;
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}
void xchg_world_rank(const mk_xchg *x, int *world, int *rank) { *world = x->world; *rank = x->rank; }

extern "C" uint64_t mk_xchg_launch_count(mk_xchg *x) { return x ? x->launches : 0; }
