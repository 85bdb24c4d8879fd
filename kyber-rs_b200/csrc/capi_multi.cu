// capi_multi.cu — the multi-device context: ONE host batch sharded over the GPUs of a box from one process.
//
// The path shards without any exchange (SURVEY §8e): signature and scalar-multiplication batches by index, DKG rounds
// by dealer.  The only data-path collective is the one the MSM needs: every device reduces its points to one
// uncompressed partial sum (128 bytes), ncclAllGather moves the partials over NVLink, every device folds them.
// One host thread per device drives that device's kb_ctx through the ordinary host-buffer entry points (so the
// copies of the shards run concurrently on all PCIe links); NCCL is bound at run time (dlopen of libnccl.so.2), so the
// library has no link-time dependency on it and single-device users never load it.
#include <dlfcn.h>
#include <nccl.h>

#include <thread>
#include <vector>

#include "ctx.cuh"

struct kb_nccl_api {
    void* lib;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    const char* (*GetErrorString)(ncclResult_t);
};

struct kb_mctx {
    int ndev;
    kb_ctx* ctx[KB_MAX_DEVICES];
    ncclComm_t comm[KB_MAX_DEVICES];
    int have_comm;
    kb_nccl_api nccl;
    uint8_t* d_part[KB_MAX_DEVICES];   // 128-byte partial of this device
    uint8_t* d_all[KB_MAX_DEVICES];    // ndev x 128 bytes gathered + 32-byte result + 8-byte bad counter
    char err[256];
};

static bool kb_nccl_load(kb_nccl_api* a)
{
    const char* names[] = {getenv("KB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm) continue;
        a->lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (a->lib) break;
    }
    if (!a->lib) return false;
    a->CommInitAll = (decltype(a->CommInitAll))dlsym(a->lib, "ncclCommInitAll");
    a->CommDestroy = (decltype(a->CommDestroy))dlsym(a->lib, "ncclCommDestroy");
    a->AllGather = (decltype(a->AllGather))dlsym(a->lib, "ncclAllGather");
    a->GroupStart = (decltype(a->GroupStart))dlsym(a->lib, "ncclGroupStart");
    a->GroupEnd = (decltype(a->GroupEnd))dlsym(a->lib, "ncclGroupEnd");
    a->GetErrorString = (decltype(a->GetErrorString))dlsym(a->lib, "ncclGetErrorString");
    return a->CommInitAll && a->CommDestroy && a->AllGather && a->GroupStart && a->GroupEnd && a->GetErrorString;
}

// contiguous, balanced [lo, hi) of n items for device i of ndev (the first n % ndev devices get one more)
static inline void kb_shard(size_t n, int i, int ndev, size_t* lo, size_t* hi)
{
    const size_t base = n / ndev, rem = n % ndev;
    *lo = (size_t)i * base + ((size_t)i < rem ? (size_t)i : rem);
    *hi = *lo + base + ((size_t)i < rem ? 1 : 0);
}

// run fn(i) on one host thread per device, return the first non-zero result
template <typename F>
static int kb_on_all(kb_mctx* m, F fn)
{
    int rc[KB_MAX_DEVICES];
    std::vector<std::thread> th;
    for (int i = 1; i < m->ndev; i++) th.emplace_back([&, i] { rc[i] = fn(i); });
    rc[0] = fn(0);
    for (auto& t : th) t.join();
    for (int i = 0; i < m->ndev; i++) {
        if (rc[i] != KB_OK) {
            snprintf(m->err, sizeof(m->err), "device %d: %s", m->ctx[i]->device, rc[i] == KB_ERR_NCCL ? m->err : kb_last_error(m->ctx[i]));
            return rc[i];
        }
    }
    return KB_OK;
}

extern "C" {

int kb_mctx_create(const int* devices, int ndev, kb_mctx** out)
{
    if (!out) return KB_ERR_ARG;
    *out = nullptr;
    if (!devices || ndev < 1 || ndev > KB_MAX_DEVICES) return KB_ERR_ARG;
    for (int i = 0; i < ndev; i++)
        for (int j = i + 1; j < ndev; j++)
            if (devices[i] == devices[j]) return KB_ERR_ARG;
    kb_mctx* m = (kb_mctx*)calloc(1, sizeof(kb_mctx));
    if (!m) return KB_ERR_NOMEM;
    m->ndev = ndev;
    int rc = KB_OK;
    for (int i = 0; i < ndev && rc == KB_OK; i++) {
        rc = kb_ctx_create(devices[i], &m->ctx[i]);
        if (rc == KB_OK) {
            if (cudaSetDevice(devices[i]) != cudaSuccess || cudaMalloc(&m->d_part[i], 128) != cudaSuccess || cudaMalloc(&m->d_all[i], 128 * (size_t)ndev + 64) != cudaSuccess) rc = KB_ERR_CUDA;
        }
    }
    if (rc == KB_OK && ndev > 1) {
        // the communicator over NVLink / NVSwitch for the MSM partials
        if (!kb_nccl_load(&m->nccl)) rc = KB_ERR_NCCL;
        else {
            const ncclResult_t r = m->nccl.CommInitAll(m->comm, ndev, devices);
            if (r != ncclSuccess) rc = KB_ERR_NCCL;
            else m->have_comm = 1;
        }
    }
    if (rc != KB_OK) {
        kb_mctx_destroy(m);
        return rc;
    }
    *out = m;
    return KB_OK;
}

void kb_mctx_destroy(kb_mctx* m)
{
    if (!m) return;
    for (int i = 0; i < m->ndev; i++) {
        if (!m->ctx[i]) continue;
        cudaSetDevice(m->ctx[i]->device);
        if (m->have_comm && m->comm[i]) m->nccl.CommDestroy(m->comm[i]);
        if (m->d_part[i]) cudaFree(m->d_part[i]);
        if (m->d_all[i]) cudaFree(m->d_all[i]);
        kb_ctx_destroy(m->ctx[i]);
    }
    free(m);
}
int kb_mctx_device_count(const kb_mctx* m) { return m ? m->ndev : 0; }
kb_ctx* kb_mctx_ctx(kb_mctx* m, int i) { return (m && i >= 0 && i < m->ndev) ? m->ctx[i] : nullptr; }
const char* kb_mctx_last_error(const kb_mctx* m) { return m ? m->err : "no context"; }
uint64_t kb_mctx_launch_count(const kb_mctx* m)
{
    uint64_t s = 0;
    if (m)
        for (int i = 0; i < m->ndev; i++) s += kb_launch_count(m->ctx[i]);
    return s;
}

// ---- sharded by index ------------------------------------------------------------------------------------------------
int kb_mctx_verify_batch(kb_mctx* m, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr)
{
    if (!m || (n && (!pk || !msg_off || !sig || !status))) return KB_ERR_ARG;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        if (hi == lo) return (int)KB_OK;
        // message offsets stay absolute: every device is handed the whole message array and its own slice of offsets
        return schnorr ? kb_schnorr_verify_batch(m->ctx[i], hi - lo, pk + 32 * lo, msg, msg_off + lo, sig + 64 * lo, status + lo)
                       : kb_eddsa_verify_batch(m->ctx[i], hi - lo, pk + 32 * lo, msg, msg_off + lo, sig + 64 * lo, status + lo);
    });
}
int kb_mctx_point_mul_base_batch(kb_mctx* m, size_t n, const uint8_t* scalars, uint8_t* out, uint32_t flags)
{
    if (!m || (n && (!scalars || !out))) return KB_ERR_ARG;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        return kb_point_mul_base_batch(m->ctx[i], hi - lo, scalars + 32 * lo, out + 32 * lo, flags);
    });
}
int kb_mctx_point_mul_batch(kb_mctx* m, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out, uint8_t* status, uint32_t flags)
{
    if (!m || (n && (!scalars || !points || !out))) return KB_ERR_ARG;
    const bool shared = (flags & KB_FLAG_SHARED_POINT) != 0;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        return kb_point_mul_batch(m->ctx[i], hi - lo, scalars + 32 * lo, shared ? points : points + 32 * lo, out + 32 * lo, status ? status + lo : nullptr, flags);
    });
}

// ---- sharded by dealer -----------------------------------------------------------------------------------------------
int kb_mctx_dkg_process_round(kb_mctx* m, size_t n, size_t t, size_t ndealers, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict,
                              const uint8_t* deal_pk, const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                              const uint8_t* resp_pk, const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status)
{
    if (!m || !t || (n && ndealers && (!commits || !shares || !verdict))) return KB_ERR_ARG;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(ndealers, i, m->ndev, &lo, &hi);
        if (hi == lo) return (int)KB_OK;
        // the commitment / share / verdict arrays are indexed by absolute dealer; the signature arrays of the call are
        // handed over as the slice that belongs to the dealer range (item (d - lo) * n + i)
        const size_t k0 = lo * n;
        return kb_dkg_process_round(m->ctx[i], n, t, lo, hi, fmt, commits, shares, verdict,
                                    deal_sig ? deal_pk + 32 * k0 : nullptr, deal_msg, deal_sig ? deal_msg_off + k0 : nullptr, deal_sig ? deal_sig + 64 * k0 : nullptr, deal_sig ? deal_status + k0 : nullptr,
                                    resp_sig ? resp_pk + 32 * k0 : nullptr, resp_msg, resp_sig ? resp_msg_off + k0 : nullptr, resp_sig ? resp_sig + 64 * k0 : nullptr, resp_sig ? resp_status + k0 : nullptr);
    });
}
int kb_mctx_dkg_verify_round(kb_mctx* m, size_t n, size_t t, size_t ndealers, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict)
{
    return kb_mctx_dkg_process_round(m, n, t, ndealers, fmt, commits, shares, verdict, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

// ---- key sets, replicated on every device ------------------------------------------------------------------------------
struct kb_mkeyset {
    kb_mctx* m;
    size_t nkeys;
    kb_keyset* ks[KB_MAX_DEVICES];   // ks[i] belongs to m->ctx[i] and holds every key
};

int kb_mctx_keyset_create(kb_mctx* m, size_t nkeys, const uint8_t* pk, kb_mkeyset** out)
{
    if (!out) return KB_ERR_ARG;
    *out = nullptr;
    if (!m || nkeys == 0 || !pk) return KB_ERR_ARG;
    kb_mkeyset* mk = (kb_mkeyset*)calloc(1, sizeof(kb_mkeyset));
    if (!mk) return KB_ERR_NOMEM;
    mk->m = m;
    mk->nkeys = nkeys;
    const int rc = kb_on_all(m, [&](int i) { return kb_keyset_create(m->ctx[i], nkeys, pk, &mk->ks[i]); });
    if (rc != KB_OK) {
        kb_mctx_keyset_destroy(mk);
        return rc;
    }
    *out = mk;
    return KB_OK;
}
void kb_mctx_keyset_destroy(kb_mkeyset* mk)
{
    if (!mk) return;
    for (int i = 0; i < mk->m->ndev; i++) kb_keyset_destroy(mk->ks[i]);
    free(mk);
}
int kb_mctx_keyset_verify_batch(kb_mkeyset* mk, size_t n, const uint32_t* key_idx, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr)
{
    if (!mk || (n && (!key_idx || !msg_off || !sig || !status))) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    uint32_t over = 0;
    for (size_t i = 0; i < n; i++) over |= (uint32_t)(key_idx[i] >= mk->nkeys);
    if (over || !kb_msg_off_ok(n, msg_off) || (msg_off[n] != msg_off[0] && !msg)) return KB_ERR_ARG;
    kb_mctx* m = mk->m;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        if (hi == lo) return (int)KB_OK;
        // the device is handed its own message bytes, with offsets made relative to the first of them
        const size_t cn = hi - lo;
        const uint64_t m0 = msg_off[lo];
        uint64_t* off = (uint64_t*)malloc(8 * (cn + 1));
        if (!off) return (int)KB_ERR_NOMEM;
        for (size_t j = 0; j <= cn; j++) off[j] = msg_off[lo + j] - m0;
        const int rc = kb_keyset_verify_batch(mk->ks[i], cn, key_idx + lo, msg ? msg + m0 : nullptr, off, sig + 64 * lo, status + lo, schnorr);
        free(off);
        return rc;
    });
}
int kb_mctx_keyset_mul_batch(kb_mkeyset* mk, size_t n, const uint32_t* key_idx, const uint8_t* scalars, uint8_t* out, uint8_t* status, uint32_t flags)
{
    if (!mk || (flags & ~KB_FLAG_VARTIME) || (n && (!key_idx || !scalars || !out))) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    uint32_t over = 0;
    for (size_t i = 0; i < n; i++) over |= (uint32_t)(key_idx[i] >= mk->nkeys);
    if (over) return KB_ERR_ARG;
    kb_mctx* m = mk->m;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        if (hi == lo) return (int)KB_OK;
        return kb_keyset_mul_batch(mk->ks[i], hi - lo, key_idx + lo, scalars + 32 * lo, out + 32 * lo, status ? status + lo : nullptr, flags);
    });
}
int kb_mctx_dkg_process_round_keyed(kb_mctx* m, const kb_mkeyset* dealers, const kb_mkeyset* verifiers, size_t n, size_t t, size_t ndealers, int fmt,
                                    const void* commits, const uint8_t* shares, uint8_t* verdict,
                                    const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                                    const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status)
{
    if (!m || !t || (n && ndealers && (!commits || !shares || !verdict))) return KB_ERR_ARG;
    // the key-set checks of kb_dkg_process_round_keyed for the whole round, before any device starts
    if ((deal_sig && !dealers) || (resp_sig && !verifiers)) return KB_ERR_ARG;
    if (dealers && (dealers->m != m || dealers->nkeys < ndealers)) return KB_ERR_ARG;
    if (verifiers && (verifiers->m != m || verifiers->nkeys < n)) return KB_ERR_ARG;
    return kb_on_all(m, [&](int i) {
        size_t lo, hi;
        kb_shard(ndealers, i, m->ndev, &lo, &hi);
        if (hi == lo) return (int)KB_OK;
        // as kb_mctx_dkg_process_round: the signature arrays are handed over as the slice of the dealer range, whose
        // dealer keys keep their absolute numbers
        const size_t k0 = lo * n;
        return kb_dkg_process_round_keyed(m->ctx[i], dealers ? dealers->ks[i] : nullptr, verifiers ? verifiers->ks[i] : nullptr, n, t, lo, hi, fmt, commits, shares, verdict,
                                          deal_msg, deal_sig ? deal_msg_off + k0 : nullptr, deal_sig ? deal_sig + 64 * k0 : nullptr, deal_sig ? deal_status + k0 : nullptr,
                                          resp_msg, resp_sig ? resp_msg_off + k0 : nullptr, resp_sig ? resp_sig + 64 * k0 : nullptr, resp_sig ? resp_status + k0 : nullptr);
    });
}

// ---- sharded by points, one collective ---------------------------------------------------------------------------------
int kb_mctx_msm(kb_mctx* m, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out32, uint64_t* bad_points)
{
    if (!m || (n && (!scalars || !points)) || !out32) return KB_ERR_ARG;
    uint64_t bad[KB_MAX_DEVICES] = {0};
    const int rc = kb_on_all(m, [&](int i) {
        kb_ctx* ctx = m->ctx[i];
        KB_CUDA(cudaSetDevice(ctx->device));
        size_t lo, hi;
        kb_shard(n, i, m->ndev, &lo, &hi);
        const size_t cn = hi - lo;
        uint8_t *d_s, *d_p;
        KB_SCRATCH(0, 32 * cn, d_s);
        KB_SCRATCH(2, 32 * cn, d_p);
        if (cn) {
            KB_H2D(d_s, scalars + 32 * lo, 32 * cn);
            KB_H2D(d_p, points + 32 * lo, 32 * cn);
        }
        uint8_t* d_res = m->d_all[i] + 128 * (size_t)m->ndev;   // 32-byte encoding, then the 8-byte counter at +32
        int r = kb_dev_msm(ctx, cn, d_s, d_p, nullptr, m->d_part[i], d_res + 32, ctx->stream);
        if (r != KB_OK) return r;
        if (m->ndev > 1) {
            // the only data-path collective: 128 bytes per device over NVLink
            const ncclResult_t nr = m->nccl.AllGather(m->d_part[i], m->d_all[i], 128, ncclUint8, m->comm[i], ctx->stream);
            if (nr != ncclSuccess) {
                snprintf(m->err, sizeof(m->err), "ncclAllGather: %s", m->nccl.GetErrorString(nr));
                return (int)KB_ERR_NCCL;
            }
            r = kb_dev_point_sum(ctx, (size_t)m->ndev, m->d_all[i], d_res, ctx->stream);
        } else {
            r = kb_dev_point_sum(ctx, 1, m->d_part[i], d_res, ctx->stream);
        }
        if (r != KB_OK) return r;
        if (i == 0) KB_D2H(out32, d_res, 32);
        KB_D2H(&bad[i], d_res + 32, 8);
        KB_SYNC();
        return (int)KB_OK;
    });
    if (rc != KB_OK) return rc;
    if (bad_points) {
        uint64_t s = 0;
        for (int i = 0; i < m->ndev; i++) s += bad[i];
        *bad_points = s;
    }
    return KB_OK;
}

}  // extern "C"
