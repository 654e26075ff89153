// host/bjj.hpp -- C++ host-side mirror of the reference crate's public API over the libbjj_cuda C ABI.
//
// The reference (arnaucube/babyjubjub-rs) is compiled Rust; this image has no Rust toolchain, so the
// host layer above include/bjj_cuda.h is provided in C++ with the reference's names, argument meaning
// and error behaviour (paths into the reference tree):
//
//   Fr                                     src/lib.rs:7     canonical 32-byte little-endian value
//   Point{x,y}::mul_scalar/compress/equals src/lib.rs:134-186
//   PointProjective{x,y,z}::affine/add     src/lib.rs:62-132
//   decompress_point / decompress_signature src/lib.rs:192-224, 260-268
//   Signature{r_b8,s}::compress            src/lib.rs:239-258
//   PrivateKey{key}::scalar_key/public/sign src/lib.rs:270-342
//   verify(pk, sig, msg)                   src/lib.rs:395-412
//   verify_schnorr(pk, m, r, s)            src/lib.rs:375-385
//   + batch entry points: mul_scalar_batch, public_batch, decompress_batch, verify_batch,
//     public_compressed_batch, sign_compressed_batch
//   + FixedBase: the comb table of a caller-chosen point, k*P and k*P + l*Q at the fixed-base rate
//   + MultiGpu: shards a batch over every device, one host thread + one bjj_ctx per device, no NCCL
//
// Header-only; link with -lbjj_cuda.  There is no CPU fallback: Engine's constructor throws when no
// CUDA device is usable.  Big integers (scalars, messages) are 32-byte little-endian arrays (U256);
// arbitrary-precision BigInt handling is the caller's job, as it is the host crate's in Rust.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../include/bjj_cuda.h"

namespace bjj_host {

using U256 = std::array<uint8_t, 32>;   // little-endian
using Fr = U256;                        // canonical field element (< Q)

inline U256 u256_from_u64(uint64_t v) {
    U256 r{};
    for (int i = 0; i < 8; i++) r[i] = (uint8_t)(v >> (8 * i));
    return r;
}

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what + ": " + bjj_error_string(c)), code(c) {}
};

class Engine {
  public:
    explicit Engine(int device = 0) {
        int rc = bjj_init(device, &ctx_);
        if (rc != BJJ_OK) throw Error(rc, "bjj_init (no CPU fallback exists)");
    }
    ~Engine() { bjj_destroy(ctx_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    bjj_ctx* ctx() const { return ctx_; }

    static void check(int rc, const char* what) {
        if (rc != BJJ_OK) throw Error(rc, what);
    }

  private:
    bjj_ctx* ctx_ = nullptr;
};

inline Engine& default_engine() {
    static Engine e(0);
    return e;
}

// ---- SoA helpers ----------------------------------------------------------------------------------
inline std::vector<uint8_t> pack(const std::vector<U256>& v) {
    std::vector<uint8_t> out(32 * v.size());
    for (size_t i = 0; i < v.size(); i++) std::memcpy(&out[32 * i], v[i].data(), 32);
    return out;
}
inline std::vector<U256> unpack(const std::vector<uint8_t>& b) {
    std::vector<U256> out(b.size() / 32);
    for (size_t i = 0; i < out.size(); i++) std::memcpy(out[i].data(), &b[32 * i], 32);
    return out;
}

struct Point;

struct PointProjective {   // src/lib.rs:62-132
    Fr x, y, z;
    Point affine(Engine& e = default_engine()) const;
    PointProjective add(const PointProjective& q, Engine& e = default_engine()) const {
        PointProjective r;
        Engine::check(bjj_add_batch(e.ctx(), 1, x.data(), y.data(), z.data(), q.x.data(), q.y.data(), q.z.data(),
                                    r.x.data(), r.y.data(), r.z.data()), "bjj_add_batch");
        return r;
    }
};

struct Point {             // src/lib.rs:134-186
    Fr x, y;
    PointProjective projective() const { return PointProjective{x, y, u256_from_u64(1)}; }
    Point mul_scalar(const U256& n, Engine& e = default_engine()) const {
        Point r;
        Engine::check(bjj_mul_scalar_batch(e.ctx(), 1, x.data(), y.data(), n.data(), r.x.data(), r.y.data()),
                      "bjj_mul_scalar_batch");
        return r;
    }
    std::array<uint8_t, 32> compress(Engine& e = default_engine()) const {
        std::array<uint8_t, 32> out;
        Engine::check(bjj_compress_batch(e.ctx(), 1, x.data(), y.data(), out.data()), "bjj_compress_batch");
        return out;
    }
    bool equals(const Point& p) const { return x == p.x && y == p.y; }
};

inline Point PointProjective::affine(Engine& e) const {
    Point r;
    Engine::check(bjj_affine_batch(e.ctx(), 1, x.data(), y.data(), z.data(), r.x.data(), r.y.data()), "bjj_affine_batch");
    return r;
}

// Result<Point, String>: throws std::invalid_argument carrying the reference's exact Err string
inline Point decompress_point(const std::array<uint8_t, 32>& bb, Engine& e = default_engine()) {   // src/lib.rs:192-224
    Point r;
    uint8_t st = 0;
    Engine::check(bjj_decompress_batch(e.ctx(), 1, bb.data(), r.x.data(), r.y.data(), &st), "bjj_decompress_batch");
    if (st) throw std::invalid_argument(bjj_status_string(st));
    return r;
}

struct Signature {         // src/lib.rs:239-258
    Point r_b8;
    U256 s;
    std::array<uint8_t, 64> compress(Engine& e = default_engine()) const {
        std::array<uint8_t, 64> out;
        auto c = r_b8.compress(e);
        std::memcpy(out.data(), c.data(), 32);
        std::memcpy(out.data() + 32, s.data(), 32);
        return out;
    }
};

inline Signature decompress_signature(const std::array<uint8_t, 64>& b, Engine& e = default_engine()) {   // src/lib.rs:260-268
    std::array<uint8_t, 32> rb;
    std::memcpy(rb.data(), b.data(), 32);
    Signature sig;
    sig.r_b8 = decompress_point(rb, e);
    std::memcpy(sig.s.data(), b.data() + 32, 32);
    return sig;
}

struct PrivateKey {        // src/lib.rs:270-342
    std::array<uint8_t, 32> key;
    static PrivateKey import(const std::vector<uint8_t>& b) {
        if (b.size() != 32) throw std::invalid_argument("imported key can not be bigger than 32 bytes");
        PrivateKey k;
        std::memcpy(k.key.data(), b.data(), 32);
        return k;
    }
    U256 scalar_key(Engine& e = default_engine()) const {
        U256 out;
        Engine::check(bjj_scalar_key_batch(e.ctx(), 1, key.data(), out.data()), "bjj_scalar_key_batch");
        return out;
    }
    Point public_key(Engine& e = default_engine()) const {   // `public` is a C++ keyword
        Point r;
        Engine::check(bjj_public_batch(e.ctx(), 1, key.data(), r.x.data(), r.y.data()), "bjj_public_batch");
        return r;
    }
    Signature sign(const U256& msg, Engine& e = default_engine()) const {
        Signature sig;
        uint8_t st = 0;
        Engine::check(bjj_sign_batch(e.ctx(), 1, key.data(), msg.data(), sig.r_b8.x.data(), sig.r_b8.y.data(),
                                     sig.s.data(), &st), "bjj_sign_batch");
        if (st) throw std::invalid_argument(bjj_status_string(st));
        return sig;
    }
};

inline bool verify(const Point& pk, const Signature& sig, const U256& msg, Engine& e = default_engine()) {   // src/lib.rs:395-412
    uint8_t ok = 0;
    Engine::check(bjj_verify_batch(e.ctx(), 1, sig.r_b8.x.data(), sig.r_b8.y.data(), sig.s.data(), pk.x.data(),
                                   pk.y.data(), msg.data(), &ok), "bjj_verify_batch");
    return ok == 1;
}

// verify_schnorr (src/lib.rs:375-385): Result<bool, String> -- throws std::invalid_argument("msg outside the
// Finite Field") for msg > Q.  `s` must already be reduced below 2^256 (the reference's s = k + x*h is an
// unreduced ~1024-bit BigInt; reduce it mod SUBORDER, the order of B8).
inline bool verify_schnorr(const Point& pk, const U256& m, const Point& r, const U256& s, Engine& e = default_engine()) {
    uint8_t ok = 0, st = 0;
    Engine::check(bjj_verify_schnorr_batch(e.ctx(), 1, pk.x.data(), pk.y.data(), m.data(), r.x.data(), r.y.data(), s.data(),
                                           &ok, &st), "bjj_verify_schnorr_batch");
    if (st) throw std::invalid_argument(bjj_status_string(st));
    return ok == 1;
}

// ---- batch entry points (the north star's additions) -------------------------------------------------
inline std::vector<Point> mul_scalar_batch(const std::vector<Point>& pts, const std::vector<U256>& scalars,
                                           Engine& e = default_engine()) {
    const size_t n = pts.size();
    std::vector<uint8_t> px(32 * n), py(32 * n), rx(32 * n), ry(32 * n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(&px[32 * i], pts[i].x.data(), 32);
        std::memcpy(&py[32 * i], pts[i].y.data(), 32);
    }
    auto k = pack(scalars);
    Engine::check(bjj_mul_scalar_batch(e.ctx(), n, px.data(), py.data(), k.data(), rx.data(), ry.data()), "bjj_mul_scalar_batch");
    std::vector<Point> out(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(out[i].x.data(), &rx[32 * i], 32);
        std::memcpy(out[i].y.data(), &ry[32 * i], 32);
    }
    return out;
}

inline std::vector<Point> public_batch(const std::vector<PrivateKey>& keys, Engine& e = default_engine()) {
    const size_t n = keys.size();
    std::vector<uint8_t> k(32 * n), rx(32 * n), ry(32 * n);
    for (size_t i = 0; i < n; i++) std::memcpy(&k[32 * i], keys[i].key.data(), 32);
    Engine::check(bjj_public_batch(e.ctx(), n, k.data(), rx.data(), ry.data()), "bjj_public_batch");
    std::vector<Point> out(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(out[i].x.data(), &rx[32 * i], 32);
        std::memcpy(out[i].y.data(), &ry[32 * i], 32);
    }
    return out;
}

// [k.public_key().compress() for k in keys] (src/lib.rs:304-306, 166-178), compressed on the device
inline std::vector<std::array<uint8_t, 32>> public_compressed_batch(const std::vector<PrivateKey>& keys,
                                                                    Engine& e = default_engine()) {
    const size_t n = keys.size();
    std::vector<uint8_t> k(32 * n), out(32 * n);
    for (size_t i = 0; i < n; i++) std::memcpy(&k[32 * i], keys[i].key.data(), 32);
    Engine::check(bjj_public_compressed_batch(e.ctx(), n, k.data(), out.data()), "bjj_public_compressed_batch");
    return unpack(out);
}

struct SignCompressedResult {
    std::array<uint8_t, 64> sig;          // compress(R8) || S; 64 zero bytes when status != 0
    uint8_t status;                       // 0 ok; otherwise bjj_status_string(status) is the reference's Err text
};
// [k.sign(m).compress() for k, m in zip(keys, msgs)] (src/lib.rs:308-342, 245-257); msg > Q gives status
// BJJ_STATUS_MSG_RANGE ("msg outside the Finite Field")
inline std::vector<SignCompressedResult> sign_compressed_batch(const std::vector<PrivateKey>& keys, const std::vector<U256>& msgs,
                                                               Engine& e = default_engine()) {
    if (keys.size() != msgs.size()) throw std::invalid_argument("keys and msgs differ in length");
    const size_t n = keys.size();
    std::vector<uint8_t> k(32 * n), sig(64 * n), st(n);
    for (size_t i = 0; i < n; i++) std::memcpy(&k[32 * i], keys[i].key.data(), 32);
    auto m = pack(msgs);
    Engine::check(bjj_sign_compressed_batch(e.ctx(), n, k.data(), m.data(), sig.data(), st.data()), "bjj_sign_compressed_batch");
    std::vector<SignCompressedResult> out(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(out[i].sig.data(), &sig[64 * i], 64);
        out[i].status = st[i];
    }
    return out;
}

// The comb table of one on-curve point P on an Engine (50 MB of device memory, freed by the destructor): P.mul_scalar(k)
// for many k at the rate of B8's fixed-base path.  Throws Error with BJJ_ERR_ARG for an off-curve P (use
// mul_scalar_batch there) and BJJ_ERR_NONCANONICAL for a coordinate >= Q.  Must not outlive its Engine.
class FixedBase {
  public:
    FixedBase(const Point& p, Engine& e = default_engine()) : e_(e) {
        Engine::check(bjj_base_create(e.ctx(), p.x.data(), p.y.data(), &base_), "bjj_base_create");
    }
    ~FixedBase() { bjj_base_destroy(e_.ctx(), base_); }
    FixedBase(const FixedBase&) = delete;
    FixedBase& operator=(const FixedBase&) = delete;
    const bjj_base* raw() const { return base_; }

    // [P.mul_scalar(k) for k in scalars]; scalars are raw 256-bit values (reduce wider ones mod ORDER)
    std::vector<Point> mul_batch(const std::vector<U256>& scalars) const {
        const size_t n = scalars.size();
        auto k = pack(scalars);
        std::vector<uint8_t> rx(32 * n), ry(32 * n);
        Engine::check(bjj_base_mul_batch(e_.ctx(), base_, n, k.data(), rx.data(), ry.data()), "bjj_base_mul_batch");
        return points(rx, ry);
    }
    // k[i]*P + l[i]*q (src/lib.rs:70-131); q == nullptr selects B8
    std::vector<Point> mul2_batch(const std::vector<U256>& k, const FixedBase* q, const std::vector<U256>& l) const {
        if (k.size() != l.size()) throw std::invalid_argument("k and l differ in length");
        const size_t n = k.size();
        auto kb = pack(k), lb = pack(l);
        std::vector<uint8_t> rx(32 * n), ry(32 * n);
        Engine::check(bjj_base_mul2_batch(e_.ctx(), base_, q ? q->raw() : nullptr, n, kb.data(), lb.data(), rx.data(), ry.data()),
                      "bjj_base_mul2_batch");
        return points(rx, ry);
    }

  private:
    static std::vector<Point> points(const std::vector<uint8_t>& rx, const std::vector<uint8_t>& ry) {
        std::vector<Point> out(rx.size() / 32);
        for (size_t i = 0; i < out.size(); i++) {
            std::memcpy(out[i].x.data(), &rx[32 * i], 32);
            std::memcpy(out[i].y.data(), &ry[32 * i], 32);
        }
        return out;
    }
    Engine& e_;
    bjj_base* base_ = nullptr;
};

struct DecompressResult {
    Point point;
    uint8_t status;                       // 0 ok; otherwise bjj_status_string(status) is the reference's Err text
};
inline std::vector<DecompressResult> decompress_batch(const std::vector<std::array<uint8_t, 32>>& blobs,
                                                      Engine& e = default_engine()) {
    const size_t n = blobs.size();
    std::vector<uint8_t> in(32 * n), rx(32 * n), ry(32 * n), st(n);
    for (size_t i = 0; i < n; i++) std::memcpy(&in[32 * i], blobs[i].data(), 32);
    Engine::check(bjj_decompress_batch(e.ctx(), n, in.data(), rx.data(), ry.data(), st.data()), "bjj_decompress_batch");
    std::vector<DecompressResult> out(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(out[i].point.x.data(), &rx[32 * i], 32);
        std::memcpy(out[i].point.y.data(), &ry[32 * i], 32);
        out[i].status = st[i];
    }
    return out;
}

inline std::vector<uint8_t> verify_batch(const std::vector<Point>& pks, const std::vector<Signature>& sigs,
                                         const std::vector<U256>& msgs, Engine& e = default_engine()) {
    const size_t n = pks.size();
    std::vector<uint8_t> r8x(32 * n), r8y(32 * n), s(32 * n), ax(32 * n), ay(32 * n), ok(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(&r8x[32 * i], sigs[i].r_b8.x.data(), 32);
        std::memcpy(&r8y[32 * i], sigs[i].r_b8.y.data(), 32);
        std::memcpy(&s[32 * i], sigs[i].s.data(), 32);
        std::memcpy(&ax[32 * i], pks[i].x.data(), 32);
        std::memcpy(&ay[32 * i], pks[i].y.data(), 32);
    }
    auto m = pack(msgs);
    Engine::check(bjj_verify_batch(e.ctx(), n, r8x.data(), r8y.data(), s.data(), ax.data(), ay.data(), m.data(), ok.data()),
                  "bjj_verify_batch");
    return ok;
}

// ---- multi-GPU: contiguous shards, one host thread + one context + one stream per device, no NCCL ------
class MultiGpu {
  public:
    MultiGpu() {
        int n = bjj_device_count();
        if (n < 1) throw Error(BJJ_ERR_CUDA, "no CUDA device (no CPU fallback exists)");
        for (int d = 0; d < n; d++) engines_.emplace_back(new Engine(d));
    }
    ~MultiGpu() {
        for (auto* e : engines_) delete e;
    }
    size_t devices() const { return engines_.size(); }

    // SoA verify over all devices; arrays are n x 32 bytes (ok: n bytes)
    void verify_batch(size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s, const uint8_t* ax,
                      const uint8_t* ay, const uint8_t* msg, uint8_t* ok) {
        shard(n, [&](Engine& e, size_t off, size_t m) {
            return bjj_verify_batch(e.ctx(), m, r8x + 32 * off, r8y + 32 * off, s + 32 * off, ax + 32 * off, ay + 32 * off,
                                    msg + 32 * off, ok + off);
        });
    }
    void mul_scalar_batch(size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* k, uint8_t* rx, uint8_t* ry) {
        shard(n, [&](Engine& e, size_t off, size_t m) {
            return bjj_mul_scalar_batch(e.ctx(), m, px + 32 * off, py + 32 * off, k + 32 * off, rx + 32 * off, ry + 32 * off);
        });
    }
    void public_batch(size_t n, const uint8_t* keys, uint8_t* rx, uint8_t* ry) {
        shard(n, [&](Engine& e, size_t off, size_t m) {
            return bjj_public_batch(e.ctx(), m, keys + 32 * off, rx + 32 * off, ry + 32 * off);
        });
    }

  private:
    template <class F>
    void shard(size_t n, F f) {
        const size_t g = engines_.size();
        std::vector<int> rc(g, BJJ_OK);
        std::vector<std::thread> th;
        for (size_t d = 0; d < g; d++) {
            const size_t off = n * d / g, end = n * (d + 1) / g;
            th.emplace_back([&, d, off, end]() { rc[d] = end > off ? f(*engines_[d], off, end - off) : BJJ_OK; });
        }
        for (auto& t : th) t.join();
        for (size_t d = 0; d < g; d++) Engine::check(rc[d], "MultiGpu shard");
    }
    std::vector<Engine*> engines_;
};

}  // namespace bjj_host
