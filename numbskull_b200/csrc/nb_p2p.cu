// Peer-to-peer halo exchange for partitioned graphs (one process per GPU).
//
// Instead of gather -> NCCL send/recv -> scatter, the owner of a boundary variable
// stores its fresh value straight into the ghost slot of every rank that holds a
// copy, through that rank's value array mapped with CUDA IPC (NVLink peer stores),
// and the ranks synchronise with a flag barrier in the same kernel: after its
// stores are fenced system-wide a rank writes the phase number into a flag word
// in each neighbour's memory and spins until all neighbours have done the same.
// One small launch per colour; no host involvement, no pack / unpack buffers.
#include <algorithm>
#include <cstring>

#include "nb_common.cuh"

struct NbP2P {
    int world = 0, rank = 0;
    std::vector<void *> opened;            // IPC mappings to close
    nb_val_t **d_peer_val[2] = {nullptr, nullptr};   // [world] device arrays of peer value arrays
    uint32_t **d_peer_flags = nullptr;     // [world] peers' flag arrays
    uint32_t *d_flags = nullptr;           // [world] my flag words, written by the peers
    int32_t *d_neigh = nullptr;            // neighbour ranks
    int n_neigh = 0;
    int32_t *d_src = nullptr, *d_peer = nullptr, *d_dst = nullptr;   // plan entries sorted by colour
    std::vector<int64_t> color_ptr;
    uint32_t *d_done = nullptr;
    int *d_error = nullptr;
    uint32_t phase = 0;
    cudaStream_t side = nullptr;           // high-priority stream of the boundary phases (split mode)
    cudaEvent_t ev_main = nullptr, ev_side = nullptr;
};

static NbP2P *p2p_of(nb_graph *g) { return (NbP2P *)g->p2p; }

extern "C" int nb_p2p_export(nb_graph *g, int world, int rank, uint8_t *handles /* 3 x 64 bytes */)
{
    NB_CUDA(cudaSetDevice(g->device));
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    // the halo moves one byte per value: graphs with cardinalities above 255 are single-GPU only
    if (g->value_bytes != 1) NB_FAIL(NB_ERR_UNSUPPORTED, "cardinalities above 255 are single-GPU only");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    if (!g->p2p) g->p2p = new NbP2P();
    NbP2P *p = p2p_of(g);
    p->world = world;
    p->rank = rank;
    if (!p->d_flags) {
        NB_CUDA(cudaMalloc(&p->d_flags, sizeof(uint32_t) * (size_t)std::max(world, 1)));
        NB_CUDA(cudaMemset(p->d_flags, 0, sizeof(uint32_t) * (size_t)std::max(world, 1)));
        NB_CUDA(cudaMalloc(&p->d_done, 4));
        NB_CUDA(cudaMemset(p->d_done, 0, 4));
        NB_CUDA(cudaMalloc(&p->d_error, 4));
        NB_CUDA(cudaMemset(p->d_error, 0, 4));
    }
    cudaIpcMemHandle_t h;
    NB_CUDA(cudaIpcGetMemHandle(&h, g->d_val[0]));
    memcpy(handles, &h, 64);
    NB_CUDA(cudaIpcGetMemHandle(&h, g->d_val[1]));
    memcpy(handles + 64, &h, 64);
    NB_CUDA(cudaIpcGetMemHandle(&h, p->d_flags));
    memcpy(handles + 128, &h, 64);
    return NB_OK;
}

// handles: world x 3 x 64 bytes (entries of non-neighbours are ignored); neighbours: ranks this
// rank exchanges values with (either direction).
extern "C" int nb_p2p_open(nb_graph *g, const uint8_t *handles, const int32_t *neighbours, int n_neigh)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p) NB_FAIL(NB_ERR_INVALID, "call nb_p2p_export first");
    std::vector<nb_val_t *> v0((size_t)p->world, nullptr), v1((size_t)p->world, nullptr);
    std::vector<uint32_t *> fl((size_t)p->world, nullptr);
    for (int i = 0; i < n_neigh; i++) {
        int r = neighbours[i];
        if (r < 0 || r >= p->world || r == p->rank) NB_FAIL(NB_ERR_INVALID, "bad neighbour rank %d", r);
        void *ptr[3];
        for (int k = 0; k < 3; k++) {
            cudaIpcMemHandle_t h;
            memcpy(&h, handles + ((size_t)r * 3 + k) * 64, 64);
            NB_CUDA(cudaIpcOpenMemHandle(&ptr[k], h, cudaIpcMemLazyEnablePeerAccess));
            p->opened.push_back(ptr[k]);
        }
        v0[(size_t)r] = (nb_val_t *)ptr[0];
        v1[(size_t)r] = (nb_val_t *)ptr[1];
        fl[(size_t)r] = (uint32_t *)ptr[2];
    }
    NB_CUDA(cudaMalloc(&p->d_peer_val[0], sizeof(void *) * (size_t)p->world));
    NB_CUDA(cudaMalloc(&p->d_peer_val[1], sizeof(void *) * (size_t)p->world));
    NB_CUDA(cudaMalloc(&p->d_peer_flags, sizeof(void *) * (size_t)p->world));
    NB_CUDA(cudaMemcpy(p->d_peer_val[0], v0.data(), sizeof(void *) * (size_t)p->world, cudaMemcpyHostToDevice));
    NB_CUDA(cudaMemcpy(p->d_peer_val[1], v1.data(), sizeof(void *) * (size_t)p->world, cudaMemcpyHostToDevice));
    NB_CUDA(cudaMemcpy(p->d_peer_flags, fl.data(), sizeof(void *) * (size_t)p->world, cudaMemcpyHostToDevice));
    NB_CUDA(cudaMalloc(&p->d_neigh, sizeof(int32_t) * (size_t)std::max(n_neigh, 1)));
    if (n_neigh) NB_CUDA(cudaMemcpy(p->d_neigh, neighbours, sizeof(int32_t) * (size_t)n_neigh, cudaMemcpyHostToDevice));
    p->n_neigh = n_neigh;
    return NB_OK;
}

// new ids of local (original) variable ids: what a peer must address in THIS rank's value arrays
extern "C" int nb_p2p_local_slots(nb_graph *g, const int32_t *local_ids, int64_t n, int32_t *slots)
{
    NB_CUDA(cudaSetDevice(g->device));
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    std::vector<int32_t> o2n((size_t)g->V);
    NB_CUDA(cudaMemcpy(o2n.data(), g->d_old2new, (size_t)g->V * 4, cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; i++) {
        if (local_ids[i] < 0 || local_ids[i] >= g->V) NB_FAIL(NB_ERR_INVALID, "local id out of range");
        slots[i] = o2n[(size_t)local_ids[i]];
    }
    return NB_OK;
}

// plan: entries grouped by colour (color_ptr has n_colors + 1 offsets); entry i copies the value of
// local variable src_local[i] into slot dst_slot[i] of rank peer[i].
extern "C" int nb_p2p_set_plan(nb_graph *g, int n_colors, const int64_t *color_ptr, const int32_t *src_local,
                               const int32_t *peer, const int32_t *dst_slot)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p) NB_FAIL(NB_ERR_INVALID, "call nb_p2p_export first");
    const int64_t n = color_ptr[n_colors];
    std::vector<int32_t> src((size_t)n);
    NB_TRY(nb_p2p_local_slots(g, src_local, n, src.data()));
    p->color_ptr.assign(color_ptr, color_ptr + n_colors + 1);
    NB_CUDA(cudaMalloc(&p->d_src, sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1)));
    NB_CUDA(cudaMalloc(&p->d_peer, sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1)));
    NB_CUDA(cudaMalloc(&p->d_dst, sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1)));
    if (n) {
        NB_CUDA(cudaMemcpy(p->d_src, src.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice));
        NB_CUDA(cudaMemcpy(p->d_peer, peer, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice));
        NB_CUDA(cudaMemcpy(p->d_dst, dst_slot, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice));
    }
    return NB_OK;
}

struct HaloArgs {
    const int32_t *src, *peer, *dst;
    int64_t beg, end;
    const nb_val_t *val0, *val1;
    nb_val_t *const *peer_val0;
    nb_val_t *const *peer_val1;
    uint32_t *const *peer_flags;
    volatile uint32_t *flags;
    const int32_t *neigh;
    int n_neigh, rank, chain_mask, wait;
    uint32_t phase;
    uint32_t *done;
    int *error;
};

__global__ void __launch_bounds__(256) k_halo_push(HaloArgs a)
{
    __shared__ bool s_last;
    for (int64_t i = a.beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.end; i += (int64_t)gridDim.x * blockDim.x) {
        const int p = a.peer[i];
        const int s = a.src[i], d = a.dst[i];
        if (a.chain_mask & 1) a.peer_val0[p][d] = a.val0[s];     // NVLink peer store
        if (a.chain_mask & 2) a.peer_val1[p][d] = a.val1[s];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(a.done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence_system();
    // ---- flag barrier with the neighbours ----
    for (int k = threadIdx.x; k < a.n_neigh; k += blockDim.x) {
        const int r = a.neigh[k];
        ((volatile uint32_t *)a.peer_flags[r])[a.rank] = a.phase;       // my arrival, in r's memory
    }
    if (a.wait) {
        for (int k = threadIdx.x; k < a.n_neigh; k += blockDim.x) {
            const int r = a.neigh[k];
            const long long t0 = clock64();
            while ((int32_t)(a.flags[r] - a.phase) < 0) {
                if (clock64() - t0 > 20000000000ll) { *a.error = 1; break; }   // ~10 s: a peer died
            }
        }
        __threadfence_system();
    }
    __syncthreads();
    if (threadIdx.x == 0) *a.done = 0;
}

// wait until every neighbour has signalled `phase` (used after a run of non-blocking exchanges)
__global__ void k_halo_wait(const volatile uint32_t *flags, const int32_t *neigh, int n_neigh, uint32_t phase, int *error)
{
    for (int k = threadIdx.x; k < n_neigh; k += blockDim.x) {
        const int r = neigh[k];
        const long long t0 = clock64();
        while ((int32_t)(flags[r] - phase) < 0) {
            if (clock64() - t0 > 20000000000ll) { *error = 1; break; }
        }
    }
    __threadfence_system();
}

// Push the boundary values of `color` (chain_mask: 1 = free chain, 2 = evidence chain, 3 = both)
// to the peers and wait for theirs.  With NB_P2P_NOWAIT (16) in chain_mask the kernel only
// signals; the sweep kernels of the next colour then wait for the neighbours' signal in their
// prologue, which takes the NVLink round trip off the critical path.  Every rank must call this
// the same number of times.
extern "C" int nb_p2p_exchange(nb_graph *g, int color, int chain_mask)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p || p->color_ptr.empty()) NB_FAIL(NB_ERR_INVALID, "p2p plan not set");
    HaloArgs a;
    a.src = p->d_src; a.peer = p->d_peer; a.dst = p->d_dst;
    const bool has = color >= 0 && color + 1 < (int)p->color_ptr.size();
    a.beg = has ? p->color_ptr[(size_t)color] : 0;
    a.end = has ? p->color_ptr[(size_t)color + 1] : 0;
    a.val0 = nb_vals<nb_val_t>(g, 0); a.val1 = nb_vals<nb_val_t>(g, 1);
    a.peer_val0 = p->d_peer_val[0]; a.peer_val1 = p->d_peer_val[1];
    a.peer_flags = p->d_peer_flags; a.flags = p->d_flags; a.neigh = p->d_neigh; a.n_neigh = p->n_neigh;
    a.rank = p->rank; a.chain_mask = chain_mask & 3; a.wait = (chain_mask & 16) ? 0 : 1;
    a.phase = ++p->phase; a.done = p->d_done; a.error = p->d_error;
    int64_t n = a.end - a.beg;
    unsigned grid = (unsigned)std::min<int64_t>(std::max<int64_t>(1, (n + 255) / 256), 148);
    k_halo_push<<<grid, 256, 0, g->stream>>>(a);
    g->launches++;
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_p2p_wait(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p || p->n_neigh == 0) return NB_OK;
    k_halo_wait<<<1, 64, 0, g->stream>>>(p->d_flags, p->d_neigh, p->n_neigh, p->phase, p->d_error);
    g->launches++;
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

// what a sweep kernel must wait for before it may read ghost values (nb_sweep.cu)
void nb_p2p_wait_args(nb_graph *g, const volatile uint32_t **flags, const int32_t **neigh, int *n_neigh, uint32_t *phase,
                      int **error)
{
    NbP2P *p = p2p_of(g);
    if (!p || p->color_ptr.empty() || g->halo_wait_off) { *n_neigh = 0; *flags = nullptr; *neigh = nullptr; *phase = 0; *error = nullptr; return; }
    *flags = p->d_flags; *neigh = p->d_neigh; *n_neigh = p->n_neigh; *phase = p->phase; *error = p->d_error;
}

// Split mode: phases 2c (boundary) and 2c + 1 (interior) of colour c run concurrently -- they are
// the same colour, so independent.  The boundary phase and its halo push go to a high-priority
// side stream, the interior phase stays on the graph's stream:
//   side:  wait(interior c-1) -> boundary c (waits for the peers' push of c-1) -> push c
//   main:  wait(boundary c-1) -> interior c
// so the push and the peers' signals travel while the interior kernel runs, and the main stream
// never stalls on the exchange.
static int sweeps_split(nb_graph *g, NbP2P *p, int64_t n_epochs, int burnin, int sample_evidence, uint64_t seed, int n_phases)
{
    if (!p->side) {
        int lo = 0, hi = 0;
        NB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        NB_CUDA(cudaStreamCreateWithPriority(&p->side, cudaStreamNonBlocking, hi));
        NB_CUDA(cudaEventCreateWithFlags(&p->ev_main, cudaEventDisableTiming));
        NB_CUDA(cudaEventCreateWithFlags(&p->ev_side, cudaEventDisableTiming));
    }
    cudaStream_t main_s = g->stream, side = p->side;
    int rc = NB_OK;
    bool first = true;
    NB_CUDA(cudaEventRecord(p->ev_main, main_s));
    for (int64_t ep = 0; ep < n_epochs && rc == NB_OK; ep++) {
        const uint64_t epoch = g->epoch_counter++;
        for (int c = 0; c < n_phases && rc == NB_OK; c += 2) {
            if (!first) NB_CUDA(cudaStreamWaitEvent(main_s, p->ev_side, 0));    // boundary of the previous colour
            NB_CUDA(cudaStreamWaitEvent(side, p->ev_main, 0));                  // interior of the previous colour
            first = false;
            g->stream = side;
            rc = nb_launch_gibbs_color(g, c, burnin, sample_evidence, seed, epoch);
            if (rc == NB_OK) rc = nb_p2p_exchange(g, c, 1 | 16);
            g->stream = main_s;
            if (rc != NB_OK) break;
            NB_CUDA(cudaEventRecord(p->ev_side, side));
            g->halo_wait_off = true;
            rc = nb_launch_gibbs_color(g, c + 1, burnin, sample_evidence, seed, epoch);
            g->halo_wait_off = false;
            if (rc != NB_OK) break;
            NB_CUDA(cudaEventRecord(p->ev_main, main_s));
        }
    }
    g->stream = main_s;
    g->halo_wait_off = false;
    if (!first) NB_CUDA(cudaStreamWaitEvent(main_s, p->ev_side, 0));
    return rc;
}

// n_epochs chromatic sweeps of a partitioned graph, launched back to back from C: per colour the
// colour's kernels and the halo push; n_colors is the GLOBAL phase count (ranks that own nothing
// of a colour still take part in its exchange).  mode: bit 0 = split-phase exchange (signal only,
// the next kernels wait in their prologue), bit 1 = the colours were split with nb_split_colors
// (n_colors counts both phases of every colour; implies bit 0).
extern "C" int nb_gibbs_sweeps_p2p(nb_graph *g, int64_t n_epochs, int burnin, int sample_evidence, uint64_t seed,
                                   int n_colors, int mode)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p || p->color_ptr.empty()) NB_FAIL(NB_ERR_INVALID, "p2p plan not set");
    if (g->has_unknown_func)
        NB_FAIL(NB_ERR_NOT_IMPLEMENTED, "Error: Factor Function %d ( used in factor %lld ) is not implemented.",
                g->unknown_func_id, (long long)g->unknown_func_factor);
    NB_TRY(nb_check_tally_room(g, burnin, n_epochs));
    const int nowait = mode & 3;
    NB_TRY(nb_refresh_inlined_weights(g));   // before the streams fork
    if (mode & 2) {
        if (n_colors & 1) NB_FAIL(NB_ERR_INVALID, "split mode needs an even phase count");
        NB_TRY(sweeps_split(g, p, n_epochs, burnin, sample_evidence, seed, n_colors));
    } else {
        for (int64_t ep = 0; ep < n_epochs; ep++) {
            const uint64_t epoch = g->epoch_counter++;
            for (int c = 0; c < n_colors; c++) {
                NB_TRY(nb_launch_gibbs_color(g, c, burnin, sample_evidence, seed, epoch));
                NB_TRY(nb_p2p_exchange(g, c, 1 | (nowait ? 16 : 0)));
            }
        }
    }
    if (nowait && n_epochs > 0) NB_TRY(nb_p2p_wait(g));
    return NB_OK;
}

extern "C" int nb_p2p_check(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    NbP2P *p = p2p_of(g);
    if (!p) return NB_OK;
    int err = 0;
    NB_CUDA(cudaMemcpyAsync(&err, p->d_error, 4, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    if (err) NB_FAIL(NB_ERR_CUDA, "peer-to-peer halo exchange timed out waiting for a neighbour rank");
    return NB_OK;
}

// Unmap the peers' memory.  Partitioned graphs are torn down in two steps -- every rank closes its
// mappings, the ranks synchronise, then each frees its own arrays (nb_graph_destroy) -- so that no
// rank frees memory a peer still has mapped.
extern "C" int nb_p2p_close(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    nb_p2p_destroy(g);
    return NB_OK;
}

void nb_p2p_destroy(nb_graph *g)
{
    NbP2P *p = p2p_of(g);
    if (!p) return;
    if (p->side) { cudaStreamSynchronize(p->side); cudaStreamDestroy(p->side); cudaEventDestroy(p->ev_main); cudaEventDestroy(p->ev_side); }
    for (void *q : p->opened) cudaIpcCloseMemHandle(q);
    cudaFree(p->d_peer_val[0]); cudaFree(p->d_peer_val[1]); cudaFree(p->d_peer_flags); cudaFree(p->d_flags);
    cudaFree(p->d_neigh); cudaFree(p->d_src); cudaFree(p->d_peer); cudaFree(p->d_dst); cudaFree(p->d_done); cudaFree(p->d_error);
    delete p;
    g->p2p = nullptr;
}
