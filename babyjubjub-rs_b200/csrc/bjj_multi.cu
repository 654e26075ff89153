// bjj_multi: ONE caller, ONE host batch, N devices of one box (include/bjj_cuda.h, "multi-device" section).
//
// BASELINE.json config 4 as written: a batch of 2^24 signatures sharded evenly across the 8 GPUs of a box, "one host
// thread and stream per device and no NCCL, because there is nothing to reduce".  A bjj_multi owns one bjj_ctx per
// device and one persistent host thread per context; a call cuts the caller's arrays into contiguous shards, hands
// shard d to thread d (which runs the ordinary host-pointer entry point on its own context, i.e. the chunked,
// double-buffered copy/compute pipeline of bjj_cuda.cu) and returns when every shard is done.  No lane ever needs a
// value of another lane, so there is no collective and no peer access on the data path.
//
// Reference items batched: verify (src/lib.rs:395-412), Point::mul_scalar (:149-164), PrivateKey::public (:304-306),
// decompress_point (:192-224), decompress_signature + verify (:260-268), the compressed outputs of
// PrivateKey::public and PrivateKey::sign (:304-306 / :308-342 with :166-178 / :245-257), and PrivateKey::sign_schnorr
// with caller nonces (:344-362).
#include <cuda_runtime.h>

#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/bjj_cuda.h"

struct bjj_multi {
    std::vector<bjj_ctx*> ctx;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    std::function<int(int)> job;      // job(d) runs shard d on ctx[d]
    unsigned long long generation = 0;
    int pending = 0;
    std::vector<int> rc;
    bool stop = false;
    bool host_register = false;       // page-lock the caller's arrays around each call
};

namespace {

void worker(bjj_multi* m, int d) {
    cudaSetDevice(bjj_device(m->ctx[d]));
    unsigned long long seen = 0;
    for (;;) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_job.wait(lk, [&] { return m->stop || m->generation != seen; });
            if (m->stop) return;
            seen = m->generation;
            job = m->job;
        }
        const int rc = job(d);
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->rc[d] = rc;
            if (--m->pending == 0) m->cv_done.notify_all();
        }
    }
}

struct HostSpan {
    const void* p;
    size_t bytes;
};

// runs f(d, off, lanes) on every device's thread over contiguous shards of n lanes; first error wins
int run_sharded(bjj_multi* m, size_t n, const std::vector<HostSpan>& spans, const std::function<int(int, size_t, size_t)>& f) {
    if (!m) return BJJ_ERR_ARG;
    if (n == 0) return BJJ_OK;
    const size_t g = m->ctx.size();
    std::vector<const void*> registered;
    if (m->host_register) {
        for (const HostSpan& s : spans)
            if (s.p && s.bytes && cudaHostRegister(const_cast<void*>(s.p), s.bytes, cudaHostRegisterPortable) == cudaSuccess)
                registered.push_back(s.p);
            else
                cudaGetLastError();      // already pinned / not registrable: copies still work, only slower
    }
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->job = [&, g, n](int d) -> int {
            const size_t off = n * (size_t)d / g, end = n * ((size_t)d + 1) / g;
            return end > off ? f(d, off, end - off) : BJJ_OK;
        };
        m->pending = (int)g;
        m->generation++;
        m->cv_job.notify_all();
        m->cv_done.wait(lk, [&] { return m->pending == 0; });
        m->job = nullptr;
    }
    for (const void* p : registered) cudaHostUnregister(const_cast<void*>(p));
    for (size_t d = 0; d < g; d++)
        if (m->rc[d] != BJJ_OK) return m->rc[d];
    return BJJ_OK;
}

}  // namespace

extern "C" {

int bjj_multi_init(int n_devices, const int* devices, bjj_multi** out) {
    if (!out) return BJJ_ERR_ARG;
    *out = nullptr;
    const int avail = bjj_device_count();
    if (avail < 1) return BJJ_ERR_CUDA;
    if (n_devices <= 0) n_devices = avail;
    bjj_multi* m = new bjj_multi();
    for (int i = 0; i < n_devices; i++) {
        const int dev = devices ? devices[i] : i;
        bjj_ctx* c = nullptr;
        const int rc = (dev >= 0 && dev < avail) ? bjj_init(dev, &c) : BJJ_ERR_ARG;
        if (rc != BJJ_OK) {
            for (bjj_ctx* x : m->ctx) bjj_destroy(x);
            delete m;
            return rc;
        }
        m->ctx.push_back(c);
    }
    m->rc.assign(m->ctx.size(), BJJ_OK);
    for (size_t d = 0; d < m->ctx.size(); d++) m->workers.emplace_back(worker, m, (int)d);
    *out = m;
    return BJJ_OK;
}

void bjj_multi_destroy(bjj_multi* m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->stop = true;
    }
    m->cv_job.notify_all();
    for (auto& t : m->workers) t.join();
    for (bjj_ctx* c : m->ctx) bjj_destroy(c);
    delete m;
}

int bjj_multi_devices(bjj_multi* m) { return m ? (int)m->ctx.size() : 0; }
bjj_ctx* bjj_multi_ctx(bjj_multi* m, int i) { return (m && i >= 0 && i < (int)m->ctx.size()) ? m->ctx[i] : nullptr; }
void bjj_multi_set_host_register(bjj_multi* m, int on) {
    if (m) m->host_register = on != 0;
}
unsigned long long bjj_multi_kernel_launches(bjj_multi* m) {
    unsigned long long t = 0;
    if (m)
        for (bjj_ctx* c : m->ctx) t += bjj_kernel_launches(c);
    return t;
}

int bjj_multi_verify_batch(bjj_multi* m, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32, const uint8_t* ax,
                           const uint8_t* ay, const uint8_t* msg32, uint8_t* ok) {
    if (!m || !r8x || !r8y || !s32 || !ax || !ay || !msg32 || !ok) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{r8x, 32 * n}, {r8y, 32 * n}, {s32, 32 * n}, {ax, 32 * n}, {ay, 32 * n}, {msg32, 32 * n}, {ok, n}},
                       [&](int d, size_t off, size_t k) {
                           const size_t o = 32 * off;
                           return bjj_verify_batch(m->ctx[d], k, r8x + o, r8y + o, s32 + o, ax + o, ay + o, msg32 + o, ok + off);
                       });
}

int bjj_multi_verify_compressed_batch(bjj_multi* m, size_t n, const uint8_t* sig64, const uint8_t* pk32, const uint8_t* msg32,
                                      uint8_t* ok, uint8_t* status) {
    if (!m || !sig64 || !pk32 || !msg32 || !ok || !status) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{sig64, 64 * n}, {pk32, 32 * n}, {msg32, 32 * n}, {ok, n}, {status, n}}, [&](int d, size_t off, size_t k) {
        return bjj_verify_compressed_batch(m->ctx[d], k, sig64 + 64 * off, pk32 + 32 * off, msg32 + 32 * off, ok + off, status + off);
    });
}

int bjj_multi_mul_scalar_batch(bjj_multi* m, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx,
                               uint8_t* ry) {
    if (!m || !px || !py || !scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{px, 32 * n}, {py, 32 * n}, {scalar32, 32 * n}, {rx, 32 * n}, {ry, 32 * n}},
                       [&](int d, size_t off, size_t k) {
                           const size_t o = 32 * off;
                           return bjj_mul_scalar_batch(m->ctx[d], k, px + o, py + o, scalar32 + o, rx + o, ry + o);
                       });
}

int bjj_multi_public_batch(bjj_multi* m, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry) {
    if (!m || !key32 || !rx || !ry) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{key32, 32 * n}, {rx, 32 * n}, {ry, 32 * n}}, [&](int d, size_t off, size_t k) {
        const size_t o = 32 * off;
        return bjj_public_batch(m->ctx[d], k, key32 + o, rx + o, ry + o);
    });
}

int bjj_multi_public_compressed_batch(bjj_multi* m, size_t n, const uint8_t* key32, uint8_t* out32) {
    if (!m || !key32 || !out32) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{key32, 32 * n}, {out32, 32 * n}}, [&](int d, size_t off, size_t k) {
        const size_t o = 32 * off;
        return bjj_public_compressed_batch(m->ctx[d], k, key32 + o, out32 + o);
    });
}

int bjj_multi_sign_compressed_batch(bjj_multi* m, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                                    uint8_t* status) {
    if (!m || !key32 || !msg32 || !sig64 || !status) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{key32, 32 * n}, {msg32, 32 * n}, {sig64, 64 * n}, {status, n}}, [&](int d, size_t off, size_t k) {
        const size_t o = 32 * off;
        return bjj_sign_compressed_batch(m->ctx[d], k, key32 + o, msg32 + o, sig64 + 2 * o, status + off);
    });
}

int bjj_multi_sign_schnorr_batch(bjj_multi* m, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                                 int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status) {
    if (!m || !key32 || !msg32 || !nonce || !rx || !ry || !s || !status) return BJJ_ERR_ARG;
    if (nonce_words < 8 || nonce_words > 64 || (nonce_words & 7)) return BJJ_ERR_ARG;
    const size_t kw = (size_t)4 * nonce_words, sw = (size_t)4 * (nonce_words + 8);     // bytes per lane of nonce and s
    return run_sharded(m, n, {{key32, 32 * n}, {msg32, 32 * n}, {nonce, kw * n}, {rx, 32 * n}, {ry, 32 * n}, {s, sw * n}, {status, n}},
                       [&](int d, size_t off, size_t k) {
                           const size_t o = 32 * off;
                           return bjj_sign_schnorr_batch(m->ctx[d], k, key32 + o, msg32 + o, nonce + kw * off, nonce_words, rx + o,
                                                         ry + o, s + sw * off, status + off);
                       });
}

int bjj_multi_fixed_base_batch(bjj_multi* m, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry) {
    if (!m || !scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{scalar32, 32 * n}, {rx, 32 * n}, {ry, 32 * n}}, [&](int d, size_t off, size_t k) {
        const size_t o = 32 * off;
        return bjj_fixed_base_batch(m->ctx[d], k, scalar32 + o, rx + o, ry + o);
    });
}

int bjj_multi_decompress_batch(bjj_multi* m, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status) {
    if (!m || !in32 || !rx || !ry || !status) return BJJ_ERR_ARG;
    return run_sharded(m, n, {{in32, 32 * n}, {rx, 32 * n}, {ry, 32 * n}, {status, n}}, [&](int d, size_t off, size_t k) {
        const size_t o = 32 * off;
        return bjj_decompress_batch(m->ctx[d], k, in32 + o, rx + o, ry + o, status + off);
    });
}

}  // extern "C"
