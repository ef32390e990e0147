// multi.cu -- the steering grid (x the frames of a batch) sharded across the GPUs of one box, behind the C ABI.
//
// Every direction's power is independent (src/dsp/mimo.cpp:121-151) and so is every frame of a batch, so G ranks are
// arranged as G_d direction groups x G_f frame groups: rank r computes direction slice r % G_d of the row-major grid for
// frame slice r // G_d of the batch, and ONE ncclAllGather per batch assembles [B][D] on every rank.  No channel sharding
// (it would reorder the channel sum the parity contract fixes).  Host batches: the ranks that share a frame slice each
// upload C / G_d channel rows of it over their own PCIe link and an all-gather over NVLink inside that group replicates
// the slice (the channel-major layout makes the concatenation the stream itself) -- chunk by chunk on a copy stream
// while the previous chunk is being computed.
//
// Two ways to form the ranks:
//   * one process per GPU (torchrun): bflk_comm_unique_id on rank 0, the caller broadcasts the 128 bytes,
//     bflk_comm_init_rank on every rank's own handle;
//   * one process, several devices (what the reference's single-process AWProcessingUnit would use):
//     bflk_group_create(cfg, device_ids, n_devices, ...) -- one host thread drives all devices, collectives inside
//     ncclGroupStart / ncclGroupEnd.
// NCCL is resolved at run time (dlopen "libnccl.so.2"): libbflk.so has no link-time dependency on it, and a process that
// already loaded NCCL (PyTorch) shares that copy.  Without NCCL the single-GPU API is unaffected and these entry points
// fail with a message.
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <mutex>

#include "bflk_internal.h"

using namespace bflk;

// ---- NCCL, resolved at run time -----------------------------------------------------------------------------
namespace {

typedef void *nccl_comm_t;
struct nccl_uid { char internal[128]; };
enum { kNcclFloat = 7, kNcclInt32 = 2, kNcclMin = 3 };   // ncclFloat32, ncclInt32, ncclMin (nccl.h)

struct Nccl {
    void *lib = nullptr;
    std::string error;
    int (*GetUniqueId)(nccl_uid *) = nullptr;
    int (*CommInitRank)(nccl_comm_t *, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*CommSplit)(nccl_comm_t, int, int, nccl_comm_t *, void *) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok() const { return lib != nullptr && error.empty(); }
};

Nccl &nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            n.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.lib) break;
        }
        if (!n.lib) {
            n.error = std::string("NCCL not found (dlopen libnccl.so.2: ") + (dlerror() ? dlerror() : "?") + ")";
            return;
        }
        auto sym = [&](const char *s) {
            void *p = dlsym(n.lib, s);
            if (!p) n.error = std::string("NCCL symbol missing: ") + s;
            return p;
        };
        n.GetUniqueId = reinterpret_cast<decltype(n.GetUniqueId)>(sym("ncclGetUniqueId"));
        n.CommInitRank = reinterpret_cast<decltype(n.CommInitRank)>(sym("ncclCommInitRank"));
        n.CommDestroy = reinterpret_cast<decltype(n.CommDestroy)>(sym("ncclCommDestroy"));
        n.CommSplit = reinterpret_cast<decltype(n.CommSplit)>(sym("ncclCommSplit"));
        n.AllGather = reinterpret_cast<decltype(n.AllGather)>(sym("ncclAllGather"));
        n.AllReduce = reinterpret_cast<decltype(n.AllReduce)>(sym("ncclAllReduce"));
        n.GroupStart = reinterpret_cast<decltype(n.GroupStart)>(sym("ncclGroupStart"));
        n.GroupEnd = reinterpret_cast<decltype(n.GroupEnd)>(sym("ncclGroupEnd"));
        n.GetErrorString = reinterpret_cast<decltype(n.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return n;
}

constexpr int kRing = 3;   // chunk buffers of the host path: upload / replicate / compute in flight

}  // namespace

// One set of a rank's map buffers.  A handle has two: the synchronous calls use set 0;
// bflk_power_map_batch_sharded_dev_submit alternates, so the kernels of batch i + 1 fill one set while the all-gather of
// batch i still reads the other.
struct MapSet {
    DevBuf<float> local;    // [nf][count] tight output of this rank's kernel when the shard is ragged
    DevBuf<float> send;     // [nf_max][per] what the all-gather sends
    DevBuf<float> gather;   // [G][nf_max][per]
    Event computed;         // the set's kernels are done (the all-gather may start)
    Event gathered;         // the set's all-gather + assembly are done (set reusable, maps complete)
};

// Created on the handle's device by init_comms, with all of its streams and events.
struct bflk_comm {
    nccl_comm_t all = nullptr;   // every rank
    nccl_comm_t sub = nullptr;   // the G_d ranks that share this rank's frame slice (== all when G_f == 1; null when G_d == 1)
    int n_ranks = 1, rank = 0, gd = 1, gf = 1, dgrp = 0, fgrp = 0;
    int planned_dirs = -1;       // grid size the direction range was set for
    MapSet sets[2];
    Stream gather_stream;        // collectives of submitted device batches
    uint64_t dev_seq = 0;
    DevBuf<float> d_all;         // [B][D] assembled maps (host variant)
    DevBuf<float> d_slice[kRing];   // [C / G_d][Tj] rows this rank uploads
    DevBuf<float> d_chunk[kRing];   // [C][Tj] replicated chunk
    DevBuf<int32_t> d_agree;
    Event ev_up[kRing], ev_done[kRing];
    Event ev_async;              // end of the last submitted (not yet waited for) host batch
    Event ev_fork;               // start of a host batch on the handle's stream: its two lanes wait for it
    int async_pending = 0;
    Stream copy_stream;
    int agreed_for_frames = -1, agreed_chunk = 0;   // chunking the ranks of a frame group agreed on
    int64_t collectives = 0;

    // ~bflk_handle and init_comms wait for the handle's streams first: once these two are done too, no work of this rank
    // still uses the communicators or the buffers
    ~bflk_comm() {
        gather_stream.sync();
        copy_stream.sync();
        if (nccl().ok()) {
            if (sub && sub != all) nccl().CommDestroy(sub);
            if (all) nccl().CommDestroy(all);
        }
    }
};

struct bflk_group {
    std::vector<bflk_handle *> hs;
    std::string error;
    ~bflk_group() {
        for (bflk_handle *h : hs) bflk_destroy(h);
    }
};

#define BFLK_NCCL(h, expr)                                                                                          \
    do {                                                                                                            \
        int _r = (expr);                                                                                            \
        if (_r != 0)                                                                                                \
            return (h)->fail(BFLK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, nccl().GetErrorString ? nccl().GetErrorString(_r) : "?", __FILE__, __LINE__); \
    } while (0)

// ---- the plan: which directions and frames a rank computes (pure arithmetic, same as bflk/shard.py) -------------
namespace {

struct Plan {
    int gd, gf, dgrp, fgrp;
    int dir_first, dir_count, dir_per;     // per = ceil(D / gd): padded slice width
    int frame_first, frame_count, frame_per;
};

bool resolve_groups(int n_ranks, int dir_groups, int *gd, int *gf) {
    int g = dir_groups > 0 ? dir_groups : (n_ranks % 2 == 0 ? 2 : 1);
    if (g < 1 || n_ranks % g) return false;
    *gd = g;
    *gf = n_ranks / g;
    return true;
}

void direction_shard(int D, int groups, int g, int *first, int *count) {
    const int base = D / groups, extra = D % groups;
    *count = base + (g < extra ? 1 : 0);
    *first = g * base + std::min(g, extra);
}

void frame_shard(int B, int groups, int g, int *first, int *count, int *per_out) {
    int per = (B + groups - 1) / groups;
    per += per & 1;                         // the kernel works on block pairs
    *first = std::min(g * per, B);
    *count = std::max(0, std::min(per, B - *first));
    if (per_out) *per_out = per;
}

Plan make_plan(int D, int B, int n_ranks, int gd, int gf, int rank) {
    Plan p{};
    p.gd = gd;
    p.gf = gf;
    p.dgrp = rank % gd;
    p.fgrp = rank / gd;
    direction_shard(D, gd, p.dgrp, &p.dir_first, &p.dir_count);
    p.dir_per = (D + gd - 1) / gd;
    frame_shard(B, gf, p.fgrp, &p.frame_first, &p.frame_count, &p.frame_per);
    p.frame_per = std::min(p.frame_per, B);
    (void)n_ranks;
    return p;
}

// gathered[G][frame_per][dir_per] (rank r = frame group r / gd, direction group r % gd) -> out[B][D]
__global__ void assemble_kernel(const float *__restrict__ gathered, int B, int D, int gd, int frame_per, int dir_per,
                                float *__restrict__ out) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const int base = D / gd, extra = D % gd;
    int dg, dl;
    if (d < extra * (base + 1)) { dg = d / (base + 1); dl = d - dg * (base + 1); }
    else { dg = extra + (d - extra * (base + 1)) / base; dl = d - (dg * base + extra); }
    for (int b = blockIdx.y; b < B; b += gridDim.y) {   // grid.y is limited to 65535
        const int fg = b / frame_per, bl = b - fg * frame_per;
        out[(size_t)b * D + d] = gathered[((size_t)(fg * gd + dg) * frame_per + bl) * dir_per + dl];
    }
}

int apply_direction_range(bflk_handle *h, const Plan &p) {
    if (h->dir_first == p.dir_first && h->dir_count == p.dir_count) return BFLK_OK;
    return bflk_set_direction_range(h, p.dir_first, p.dir_count);
}

int check_sharded(bflk_handle *h, const char *who) {
    if (!h->comm) return h->fail(BFLK_ERR_STATE, "%s: the handle is not part of a multi-GPU job (bflk_comm_init_rank / bflk_group_create)", who);
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "%s: set geometry and grid first", who);
    return BFLK_OK;
}

// local compute of one rank: its direction slice of frames [f0, f0 + nf) of a device-resident stream into set.send
int compute_shard(bflk_handle *h, const Plan &p, MapSet &set, const float *stream_dev, int64_t row_stride, int64_t n_samples,
                  int f_rel0, int nf, int out_row0, const Launch &launch) {
    if (nf <= 0 || p.dir_count <= 0) return BFLK_OK;
    const int N = h->cfg.frame_len;
    const bool tight = p.dir_count == p.dir_per;
    float *out = tight ? set.send.p + (size_t)out_row0 * p.dir_per : set.local.p + (size_t)out_row0 * p.dir_count;
    int rc = power_map_dev(h, stream_dev + (size_t)f_rel0 * N, row_stride, n_samples - (int64_t)f_rel0 * N, nf, out, launch);
    if (rc) return rc;
    if (!tight)
        BFLK_CUDA(h, cudaMemcpy2DAsync(set.send.p + (size_t)out_row0 * p.dir_per, (size_t)p.dir_per * sizeof(float), out,
                                       (size_t)p.dir_count * sizeof(float), (size_t)p.dir_count * sizeof(float), nf,
                                       cudaMemcpyDeviceToDevice, launch.st));
    return BFLK_OK;
}

int reserve_maps(bflk_handle *h, const Plan &p, MapSet &set, int B, bool need_all) {
    bflk_comm *c = h->comm;
    const size_t slice = (size_t)p.frame_per * p.dir_per;
    const bool grows = slice > set.send.n || slice * c->n_ranks > set.gather.n ||
                       (p.dir_count != p.dir_per && (size_t)p.frame_per * p.dir_count > set.local.n);
    if (grows) BFLK_CUDA(h, cudaEventSynchronize(set.gathered));   // a submitted batch may still use the set
    BFLK_CUDA(h, set.send.reserve(slice));
    BFLK_CUDA(h, set.gather.reserve(slice * c->n_ranks));
    if (p.dir_count != p.dir_per) BFLK_CUDA(h, set.local.reserve((size_t)p.frame_per * p.dir_count));
    if (need_all) BFLK_CUDA(h, c->d_all.reserve((size_t)B * h->n_dir));
    return BFLK_OK;
}

// one all-gather of the ranks' slices + assembly into out_dev[B][D]; hs = the local handles of the job (1 per process,
// or all of them in a single-process group), sets[i] = the map set handle i uses
int gather_and_assemble(const std::vector<bflk_handle *> &hs, const std::vector<Plan> &plans, const std::vector<MapSet *> &sets,
                        int B, const std::vector<float *> &out_dev, const std::vector<cudaStream_t> &st) {
    Nccl &n = nccl();
    n.GroupStart();
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_handle *h = hs[i];
        bflk_comm *c = h->comm;
        cudaSetDevice(h->cfg.device);
        const size_t slice = (size_t)plans[i].frame_per * plans[i].dir_per;
        int r = n.AllGather(sets[i]->send.p, sets[i]->gather.p, slice, kNcclFloat, c->all, st[i]);
        if (r != 0) {
            n.GroupEnd();
            return h->fail(BFLK_ERR_CUDA, "ncclAllGather failed: %s", n.GetErrorString(r));
        }
        c->collectives++;
    }
    int r = n.GroupEnd();
    if (r != 0) return hs[0]->fail(BFLK_ERR_CUDA, "ncclGroupEnd failed: %s", n.GetErrorString(r));
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_handle *h = hs[i];
        if (!out_dev[i]) continue;
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        const Plan &p = plans[i];
        dim3 grid((h->n_dir + 255) / 256, std::min(B, 65535));
        assemble_kernel<<<grid, 256, 0, st[i]>>>(sets[i]->gather.p, B, h->n_dir, p.gd, p.frame_per, p.dir_per, out_dev[i]);
        BFLK_CUDA(h, cudaGetLastError());
        h->launches++;
    }
    return BFLK_OK;
}

// pipelined = false: everything on st (the maps are complete in stream order).  pipelined = true (one handle per process):
// the kernels go on st, the all-gather + assembly on the communicator's own stream, in alternating buffer sets, so the
// kernels of the next submitted batch run under this batch's collective; sharded_dev_join makes a stream wait for them.
int sharded_dev(const std::vector<bflk_handle *> &hs, const std::vector<const float *> &stream_dev, int64_t n_samples,
                int32_t n_frames, const std::vector<float *> &power_all_dev, const std::vector<cudaStream_t> &st, bool pipelined = false) {
    std::vector<Plan> plans(hs.size());
    std::vector<MapSet *> sets(hs.size());
    std::vector<cudaStream_t> gst = st;
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_handle *h = hs[i];
        int rc = check_sharded(h, "bflk_power_map_batch_sharded_dev");
        if (rc) return rc;
        if (!stream_dev[i] || !power_all_dev[i] || n_frames <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_sharded_dev: null buffer or no frames");
        if (n_samples < min_stream_samples(h, n_frames))
            return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_sharded_dev: %lld samples per channel cannot hold %d frames", (long long)n_samples, n_frames);
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        bflk_comm *c = h->comm;
        if (pipelined) {
            sets[i] = &c->sets[c->dev_seq++ & 1];
            gst[i] = c->gather_stream;
            // the batch that used this set two submits ago: its collective must be done before the kernels overwrite the set
            BFLK_CUDA(h, cudaStreamWaitEvent(st[i], sets[i]->gathered, 0));
        } else {
            // a synchronous call after submitted batches: set 0 may still be in flight on the communicator's stream
            sets[i] = &c->sets[0];
            for (MapSet &s : c->sets) BFLK_CUDA(h, cudaStreamWaitEvent(st[i], s.gathered, 0));
        }
        plans[i] = make_plan(h->n_dir, n_frames, c->n_ranks, c->gd, c->gf, c->rank);
        if ((rc = apply_direction_range(h, plans[i]))) return rc;
        if ((rc = reserve_maps(h, plans[i], *sets[i], n_frames, false))) return rc;
        // The kernels stay on the caller's stream.  Alternating them between the handle's two lanes as well
        // (power_map_dev_overlapped) was measured and not kept: +1.6 % on two GPUs (149.4 k vs 147.0 k maps/s) but -7.7 % on
        // eight (529.6 k vs 573.7 k): with two buffer sets, batch i + 2 waits for the all-gather of batch i, which waits for
        // kernels that then share the SMs with batch i + 1 -- a bubble per batch once a launch is only four waves.
        if ((rc = compute_shard(h, plans[i], *sets[i], stream_dev[i], n_samples, n_samples, plans[i].frame_first,
                                plans[i].frame_count, 0, Launch{st[i]}))) return rc;
        if (pipelined) {
            BFLK_CUDA(h, cudaEventRecord(sets[i]->computed, st[i]));
            BFLK_CUDA(h, cudaStreamWaitEvent(c->gather_stream, sets[i]->computed, 0));
        }
    }
    int rc = gather_and_assemble(hs, plans, sets, n_frames, power_all_dev, gst);
    if (pipelined && rc == BFLK_OK) {
        for (size_t i = 0; i < hs.size(); i++) {
            BFLK_CUDA(hs[i], cudaSetDevice(hs[i]->cfg.device));
            BFLK_CUDA(hs[i], cudaEventRecord(sets[i]->gathered, hs[i]->comm->gather_stream));
        }
    }
    return rc;
}

int sharded_dev_join(bflk_handle *h, cudaStream_t st) {
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    for (MapSet &s : h->comm->sets) BFLK_CUDA(h, cudaStreamWaitEvent(st, s.gathered, 0));
    return BFLK_OK;
}

// the ranks of a frame group must cut their slice into the same chunks (the input all-gather is a collective): each
// proposes the wave-aligned chunk of its own direction slice, the smallest proposal wins; agreed once per batch size
int agree_on_chunk(const std::vector<bflk_handle *> &hs, const std::vector<Plan> &plans) {
    Nccl &n = nccl();
    bool need = false;
    for (size_t i = 0; i < hs.size(); i++) need |= hs[i]->comm->agreed_for_frames != plans[i].frame_count;
    if (!need) return BFLK_OK;
    std::vector<int32_t> prop(hs.size());
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_handle *h = hs[i];
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        int cf = 1 << 30;   // a rank without frames (tiny batch) does not constrain the others
        if (plans[i].frame_count > 0) {
            int rc = host_chunk_frames(h, plans[i].frame_count, &cf);
            if (rc) return rc;
        }
        prop[i] = cf;
        BFLK_CUDA(h, h->comm->d_agree.reserve(2));
        BFLK_CUDA(h, cudaMemcpyAsync(h->comm->d_agree.p, &prop[i], sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    }
    n.GroupStart();
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_comm *c = hs[i]->comm;
        cudaSetDevice(hs[i]->cfg.device);
        n.AllReduce(c->d_agree.p, c->d_agree.p + 1, 1, kNcclInt32, kNcclMin, c->all, hs[i]->stream);
    }
    int r = n.GroupEnd();
    if (r != 0) return hs[0]->fail(BFLK_ERR_CUDA, "ncclAllReduce (chunk agreement) failed: %s", n.GetErrorString(r));
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_handle *h = hs[i];
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        int32_t v = 0;
        BFLK_CUDA(h, cudaMemcpyAsync(&v, h->comm->d_agree.p + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
        h->comm->agreed_chunk = std::max(2, (int)v);
        h->comm->agreed_for_frames = plans[i].frame_count;
    }
    return BFLK_OK;
}

int sharded_host(const std::vector<bflk_handle *> &hs, const float *stream, int64_t n_samples, int32_t n_frames,
                 const std::vector<float *> &power_out, bool wait_for_it = true) {
    Nccl &n = nccl();
    const size_t G = hs.size();
    std::vector<Plan> plans(G);
    std::vector<MapSet *> sets(G);
    for (size_t i = 0; i < G; i++) {
        bflk_handle *h = hs[i];
        int rc = check_sharded(h, "bflk_power_map_batch_sharded");
        if (rc) return rc;
        if (!stream || n_frames <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_sharded: null buffer or no frames");
        if (n_samples < min_stream_samples(h, n_frames))
            return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_sharded: %lld samples per channel cannot hold %d frames", (long long)n_samples, n_frames);
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        bflk_comm *c = h->comm;
        sets[i] = &c->sets[0];
        for (MapSet &s : c->sets)   // device batches submitted earlier may still use buffer set 0 on the communicator's stream
            BFLK_CUDA(h, cudaStreamWaitEvent(h->stream, s.gathered, 0));
        plans[i] = make_plan(h->n_dir, n_frames, c->n_ranks, c->gd, c->gf, c->rank);
        if ((rc = apply_direction_range(h, plans[i]))) return rc;
        if ((rc = reserve_maps(h, plans[i], *sets[i], n_frames, true))) return rc;
    }
    int rc = agree_on_chunk(hs, plans);
    if (rc) return rc;
    const int N = hs[0]->cfg.frame_len, C = hs[0]->cfg.n_channels;
    const int64_t tail = frame_tail_samples(hs[0]);
    // chunk j of local rank i: first sample t0 in the caller's stream, Tj valid samples per row, rows `pitch` floats apart on
    // the device (even: the tiled kernel packs with 8-byte loads)
    struct Chunk { int a, nfj; int64_t t0, Tj, pitch; };
    auto chunk_of = [&](size_t i, int j) {
        Chunk k;
        const int cf = hs[i]->comm->agreed_chunk;
        k.a = j * cf;
        k.nfj = std::min(cf, plans[i].frame_count - k.a);
        k.t0 = (int64_t)(plans[i].frame_first + k.a) * N;
        k.Tj = std::min<int64_t>((int64_t)k.nfj * N + tail, n_samples - k.t0);
        k.pitch = (k.Tj + 1) & ~(int64_t)1;
        return k;
    };
    // the chunk loop runs max-over-local-ranks iterations; a rank whose slice is exhausted (ragged last frame group) only
    // takes part in the collectives of its own frame group, which has the same chunk count by construction
    int max_chunks = 0;
    std::vector<int> n_chunks(G);
    for (size_t i = 0; i < G; i++) {
        const int cf = hs[i]->comm->agreed_chunk;
        n_chunks[i] = plans[i].frame_count > 0 ? (plans[i].frame_count + cf - 1) / cf : 0;
        max_chunks = std::max(max_chunks, n_chunks[i]);
        const int64_t Tj = (int64_t)std::min(cf, std::max(1, plans[i].frame_count)) * N + tail + 1;
        bflk_comm *c = hs[i]->comm;
        BFLK_CUDA(hs[i], cudaSetDevice(hs[i]->cfg.device));
        const bool split = c->gd > 1 && C % c->gd == 0;
        for (int k = 0; k < std::min(kRing, std::max(1, n_chunks[i])); k++) {
            BFLK_CUDA(hs[i], c->d_chunk[k].reserve((size_t)C * Tj));
            if (split) BFLK_CUDA(hs[i], c->d_slice[k].reserve((size_t)(C / c->gd) * Tj));
        }
    }
    // the chunks' kernels alternate between the handle's two lanes (own scratch each, bflk_api.cu host_chunks): the CTAs of
    // chunk j + 1 fill the SMs that the last CTAs of chunk j leave idle one by one.  Both lanes start after whatever the
    // handle's stream has queued (the previous batch's all-gather reads the buffers this batch writes).
    std::vector<char> lanes(G, 0);
    for (size_t i = 0; i < G; i++) {
        bflk_handle *h = hs[i];
        lanes[i] = n_chunks[i] > 1;
        if (!lanes[i]) continue;
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        BFLK_CUDA(h, cudaEventRecord(h->comm->ev_fork, h->stream));
        if ((rc = lanes_fork(h, h->comm->ev_fork))) return rc;
    }
    for (int j = 0; j < max_chunks; j++) {
        const int buf = j % kRing;
        // upload this chunk's rows (copy stream), after the compute that last used the buffer
        for (size_t i = 0; i < G; i++) {
            if (j >= n_chunks[i]) continue;
            bflk_handle *h = hs[i];
            bflk_comm *c = h->comm;
            BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
            const Chunk k = chunk_of(i, j);
            // the compute that last used this ring buffer (an earlier chunk of this batch, or of the previous batch when
            // batches are submitted back to back) must be done before the copy overwrites it
            BFLK_CUDA(h, cudaStreamWaitEvent(c->copy_stream, c->ev_done[buf], 0));
            const bool split = c->gd > 1 && C % c->gd == 0;
            if (split) {
                const int rows = C / c->gd;
                BFLK_CUDA(h, cudaMemcpy2DAsync(c->d_slice[buf].p, k.pitch * sizeof(float), stream + (size_t)c->dgrp * rows * n_samples + k.t0,
                                               n_samples * sizeof(float), k.Tj * sizeof(float), rows, cudaMemcpyHostToDevice, c->copy_stream));
            } else {
                BFLK_CUDA(h, cudaMemcpy2DAsync(c->d_chunk[buf].p, k.pitch * sizeof(float), stream + k.t0, n_samples * sizeof(float),
                                               k.Tj * sizeof(float), C, cudaMemcpyHostToDevice, c->copy_stream));
            }
        }
        // replicate inside each frame group over NVLink
        bool any_split = false;
        for (size_t i = 0; i < G; i++) any_split |= j < n_chunks[i] && hs[i]->comm->gd > 1 && C % hs[i]->comm->gd == 0;
        if (any_split) {
            n.GroupStart();
            for (size_t i = 0; i < G; i++) {
                if (j >= n_chunks[i]) continue;
                bflk_handle *h = hs[i];
                bflk_comm *c = h->comm;
                if (!(c->gd > 1 && C % c->gd == 0)) continue;
                cudaSetDevice(h->cfg.device);
                const Chunk k = chunk_of(i, j);
                int r = n.AllGather(c->d_slice[buf].p, c->d_chunk[buf].p, (size_t)(C / c->gd) * k.pitch, kNcclFloat, c->sub, c->copy_stream);
                if (r != 0) {
                    n.GroupEnd();
                    return h->fail(BFLK_ERR_CUDA, "ncclAllGather (input) failed: %s", n.GetErrorString(r));
                }
                c->collectives++;
            }
            int r = n.GroupEnd();
            if (r != 0) return hs[0]->fail(BFLK_ERR_CUDA, "ncclGroupEnd failed: %s", n.GetErrorString(r));
        }
        // compute the chunk
        for (size_t i = 0; i < G; i++) {
            if (j >= n_chunks[i]) continue;
            bflk_handle *h = hs[i];
            bflk_comm *c = h->comm;
            BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
            const Chunk k = chunk_of(i, j);
            cudaStream_t cs = lanes[i] ? h->lane[j & 1] : h->stream;
            BFLK_CUDA(h, cudaEventRecord(c->ev_up[buf], c->copy_stream));
            BFLK_CUDA(h, cudaStreamWaitEvent(cs, c->ev_up[buf], 0));
            rc = compute_shard(h, plans[i], *sets[i], c->d_chunk[buf].p, k.pitch, k.Tj, 0, k.nfj, k.a,
                               Launch{cs, lanes[i] ? (j & 1) : 0, (bool)lanes[i]});
            if (rc) return rc;
            BFLK_CUDA(h, cudaEventRecord(c->ev_done[buf], cs));
        }
    }
    for (size_t i = 0; i < G; i++) {   // the all-gather on the handle's stream follows every chunk
        if (!lanes[i]) continue;
        BFLK_CUDA(hs[i], cudaSetDevice(hs[i]->cfg.device));
        if ((rc = lanes_join(hs[i]))) return rc;
    }
    std::vector<float *> out_dev(G);
    std::vector<cudaStream_t> st(G);
    for (size_t i = 0; i < G; i++) {
        out_dev[i] = power_out[i] ? hs[i]->comm->d_all.p : nullptr;
        st[i] = hs[i]->stream;
    }
    if ((rc = gather_and_assemble(hs, plans, sets, n_frames, out_dev, st))) return rc;
    for (size_t i = 0; i < G; i++) {
        bflk_handle *h = hs[i];
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        if (power_out[i])
            BFLK_CUDA(h, cudaMemcpyAsync(power_out[i], h->comm->d_all.p, (size_t)n_frames * h->n_dir * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    }
    for (size_t i = 0; i < G; i++) {
        bflk_handle *h = hs[i];
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        if (wait_for_it) {
            BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
            h->comm->async_pending = 0;
        } else {
            BFLK_CUDA(h, cudaEventRecord(h->comm->ev_async, h->stream));   // everything of this batch precedes it on the stream
            h->comm->async_pending++;
        }
    }
    return BFLK_OK;
}

int init_comms(const std::vector<bflk_handle *> &hs, const std::vector<int> &ranks, const nccl_uid &id, int n_ranks, int dir_groups) {
    Nccl &n = nccl();
    int gd = 1, gf = 1;
    if (!resolve_groups(n_ranks, dir_groups, &gd, &gf))
        return hs[0]->fail(BFLK_ERR_INVALID, "bflk_comm_init: %d direction groups do not divide %d ranks", dir_groups, n_ranks);
    for (bflk_handle *h : hs) {
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        BFLK_CUDA(h, cudaStreamSynchronize(h->stream));   // the collectives of the old communicator are done
        comm_release(h);
        cudaGetLastError();   // clear an earlier call's error: the check below is about the new streams and events
        h->comm = new bflk_comm();
        BFLK_CUDA(h, cudaGetLastError());
    }
    n.GroupStart();
    for (size_t i = 0; i < hs.size(); i++) {
        bflk_comm *c = hs[i]->comm;
        c->n_ranks = n_ranks;
        c->rank = ranks[i];
        c->gd = gd;
        c->gf = gf;
        c->dgrp = ranks[i] % gd;
        c->fgrp = ranks[i] / gd;
        cudaSetDevice(hs[i]->cfg.device);
        int r = n.CommInitRank(&c->all, n_ranks, id, ranks[i]);
        if (r != 0) {
            n.GroupEnd();
            return hs[i]->fail(BFLK_ERR_CUDA, "ncclCommInitRank failed: %s", n.GetErrorString(r));
        }
    }
    int r = n.GroupEnd();
    if (r != 0) return hs[0]->fail(BFLK_ERR_CUDA, "ncclCommInitRank (group) failed: %s", n.GetErrorString(r));
    if (gd > 1 && gf > 1) {
        n.GroupStart();
        for (size_t i = 0; i < hs.size(); i++) {
            bflk_comm *c = hs[i]->comm;
            cudaSetDevice(hs[i]->cfg.device);
            int rr = n.CommSplit(c->all, c->fgrp, c->dgrp, &c->sub, nullptr);
            if (rr != 0) {
                n.GroupEnd();
                return hs[i]->fail(BFLK_ERR_CUDA, "ncclCommSplit failed: %s", n.GetErrorString(rr));
            }
        }
        r = n.GroupEnd();
        if (r != 0) return hs[0]->fail(BFLK_ERR_CUDA, "ncclCommSplit (group) failed: %s", n.GetErrorString(r));
    } else if (gd > 1) {
        for (bflk_handle *h : hs) h->comm->sub = h->comm->all;
    }
    return BFLK_OK;
}

}  // namespace

void bflk::comm_release(bflk_handle *h) {
    delete h->comm;
    h->comm = nullptr;
}

extern "C" {

int bflk_shard_plan(int32_t n_directions, int32_t n_frames, int32_t n_ranks, int32_t dir_groups, int32_t rank,
                    int32_t *dir_first, int32_t *dir_count, int32_t *frame_first, int32_t *frame_count) {
    int gd = 1, gf = 1;
    if (n_directions <= 0 || n_frames <= 0 || n_ranks <= 0 || rank < 0 || rank >= n_ranks || !resolve_groups(n_ranks, dir_groups, &gd, &gf))
        return BFLK_ERR_INVALID;
    const Plan p = make_plan(n_directions, n_frames, n_ranks, gd, gf, rank);
    if (dir_first) *dir_first = p.dir_first;
    if (dir_count) *dir_count = p.dir_count;
    if (frame_first) *frame_first = p.frame_first;
    if (frame_count) *frame_count = p.frame_count;
    return BFLK_OK;
}

int bflk_comm_unique_id(uint8_t *id128) {
    if (!id128) return BFLK_ERR_INVALID;
    if (!nccl().ok()) return BFLK_ERR_STATE;
    nccl_uid id;
    if (nccl().GetUniqueId(&id) != 0) return BFLK_ERR_CUDA;
    std::memcpy(id128, id.internal, 128);
    return BFLK_OK;
}

int bflk_comm_init_rank(bflk_handle *h, const uint8_t *id128, int32_t n_ranks, int32_t rank, int32_t dir_groups) {
    if (!h) return BFLK_ERR_INVALID;
    if (!id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return h->fail(BFLK_ERR_INVALID, "bflk_comm_init_rank: bad rank %d of %d", rank, n_ranks);
    if (!nccl().ok()) return h->fail(BFLK_ERR_STATE, "bflk_comm_init_rank: %s", nccl().error.c_str());
    nccl_uid id;
    std::memcpy(id.internal, id128, 128);
    return init_comms({h}, {rank}, id, n_ranks, dir_groups);
}

int bflk_comm_info(const bflk_handle *h, int32_t *n_ranks, int32_t *rank, int32_t *dir_groups, int32_t *frame_groups, int64_t *collectives) {
    if (!h || !h->comm) return BFLK_ERR_STATE;
    if (n_ranks) *n_ranks = h->comm->n_ranks;
    if (rank) *rank = h->comm->rank;
    if (dir_groups) *dir_groups = h->comm->gd;
    if (frame_groups) *frame_groups = h->comm->gf;
    if (collectives) *collectives = h->comm->collectives;
    return BFLK_OK;
}

int bflk_power_map_batch_sharded_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                     float *power_all_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    return sharded_dev({h}, {stream_dev}, n_samples, n_frames, {power_all_dev}, {cuda_stream ? (cudaStream_t)cuda_stream : h->stream});
}

// Continuous operation on device-resident streams: the kernels of batch i + 1 (on cuda_stream) run under the all-gather and
// assembly of batch i (on the communicator's own stream, alternating buffer sets); power_all_dev of every submitted batch is
// complete for work enqueued on cuda_stream after _join.  Collective: every rank submits and joins alike.
int bflk_power_map_batch_sharded_dev_submit(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                            float *power_all_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    return sharded_dev({h}, {stream_dev}, n_samples, n_frames, {power_all_dev}, {cuda_stream ? (cudaStream_t)cuda_stream : h->stream}, true);
}

int bflk_power_map_batch_sharded_dev_join(bflk_handle *h, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    int rc = check_sharded(h, "bflk_power_map_batch_sharded_dev_join");
    if (rc) return rc;
    return sharded_dev_join(h, cuda_stream ? (cudaStream_t)cuda_stream : h->stream);
}

int bflk_power_map_batch_sharded(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    return sharded_host({h}, stream, n_samples, n_frames, {power_out});
}

// Continuous operation: enqueue and return; the stream orders successive batches (the ring buffers of the upload path
// are guarded by events), so the uploads of batch i + 1 run under the kernels and collectives of batch i.  _wait blocks
// until everything submitted so far has delivered its maps.  Collective: every rank submits and waits alike.
int bflk_power_map_batch_sharded_submit(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    return sharded_host({h}, stream, n_samples, n_frames, {power_out}, false);
}

int bflk_power_map_batch_sharded_wait(bflk_handle *h) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->comm || h->comm->async_pending == 0) return BFLK_OK;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    BFLK_CUDA(h, cudaEventSynchronize(h->comm->ev_async));
    h->comm->async_pending = 0;
    return BFLK_OK;
}

// ---- one process, several devices -----------------------------------------------------------------------------
int bflk_group_create(const bflk_config *cfg, const int32_t *device_ids, int32_t n_devices, int32_t dir_groups, bflk_group **out) {
    if (!cfg || !device_ids || n_devices < 1 || !out) return BFLK_ERR_INVALID;
    *out = nullptr;
    std::unique_ptr<bflk_group> g(new bflk_group());
    for (int i = 0; i < n_devices; i++) {
        bflk_config c = *cfg;
        c.device = device_ids[i];
        bflk_handle *h = nullptr;
        int rc = bflk_create(&c, &h);
        if (rc) return rc;
        g->hs.push_back(h);
    }
    if (n_devices > 1) {
        if (!nccl().ok()) return BFLK_ERR_STATE;
        nccl_uid id;
        std::vector<int> ranks(n_devices);
        for (int i = 0; i < n_devices; i++) ranks[i] = i;
        int rc = nccl().GetUniqueId(&id) == 0 ? init_comms(g->hs, ranks, id, n_devices, dir_groups) : BFLK_ERR_CUDA;
        if (rc) return rc;
    }
    *out = g.release();
    return BFLK_OK;
}

int bflk_group_destroy(bflk_group *g) {
    if (!g) return BFLK_ERR_INVALID;
    delete g;
    return BFLK_OK;
}

int32_t bflk_group_size(const bflk_group *g) { return g ? (int32_t)g->hs.size() : 0; }

bflk_handle *bflk_group_handle(bflk_group *g, int32_t i) { return g && i >= 0 && i < (int32_t)g->hs.size() ? g->hs[i] : nullptr; }

const char *bflk_group_last_error(const bflk_group *g) {
    if (!g) return "";
    for (bflk_handle *h : g->hs)
        if (!h->error.empty()) return h->error.c_str();
    return g->error.c_str();
}

#define BFLK_FORALL(g, call)                       \
    do {                                           \
        if (!(g)) return BFLK_ERR_INVALID;         \
        for (bflk_handle * h : (g)->hs) {          \
            int _rc = (call);                      \
            if (_rc) return _rc;                   \
        }                                          \
        return BFLK_OK;                            \
    } while (0)

int bflk_group_set_geometry(bflk_group *g, const float *xyz, int32_t n_channels) { BFLK_FORALL(g, bflk_set_geometry(h, xyz, n_channels)); }
int bflk_group_set_tiled_geometry(bflk_group *g, int32_t n_tiles, const float *origins) { BFLK_FORALL(g, bflk_set_tiled_geometry(h, n_tiles, origins)); }
int bflk_group_set_channel_mask(bflk_group *g, const int32_t *index, int32_t usable) { BFLK_FORALL(g, bflk_set_channel_mask(h, index, usable)); }
int bflk_group_set_grid_fov(bflk_group *g, int32_t rows, int32_t cols, float fov_deg) { BFLK_FORALL(g, bflk_set_grid_fov(h, rows, cols, fov_deg)); }
int bflk_group_set_kernel(bflk_group *g, int32_t which) { BFLK_FORALL(g, bflk_set_kernel(h, which)); }

int bflk_group_power_map_batch(bflk_group *g, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!g || g->hs.empty()) return BFLK_ERR_INVALID;
    if (g->hs.size() == 1) return bflk_power_map_batch(g->hs[0], stream, n_samples, n_frames, power_out);
    std::vector<float *> outs(g->hs.size(), nullptr);
    outs[0] = power_out;   // one process: one host copy of the maps, from device 0
    return sharded_host(g->hs, stream, n_samples, n_frames, outs);
}

int bflk_group_power_map_batch_dev(bflk_group *g, const float *const *stream_dev, int64_t n_samples, int32_t n_frames,
                                   float *const *power_all_dev) {
    if (!g || g->hs.empty() || !stream_dev || !power_all_dev) return BFLK_ERR_INVALID;
    if (g->hs.size() == 1) return bflk_power_map_batch_dev(g->hs[0], stream_dev[0], n_samples, n_frames, power_all_dev[0], nullptr);
    std::vector<const float *> in(stream_dev, stream_dev + g->hs.size());
    std::vector<float *> out(power_all_dev, power_all_dev + g->hs.size());
    std::vector<cudaStream_t> st;
    for (bflk_handle *h : g->hs) st.push_back(h->stream);
    return sharded_dev(g->hs, in, n_samples, n_frames, out, st);
}

int bflk_group_synchronize(bflk_group *g) {
    if (!g) return BFLK_ERR_INVALID;
    for (bflk_handle *h : g->hs) {
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    return BFLK_OK;
}

}  // extern "C"
