// N-API addon: the thin shim between the reference's TypeScript host and libzkr's C-ABI.
// SOURCE ONLY in this repository -- node and node_api.h are not present in the build image, so this
// file is only syntax-checked here against a declarations-only stub of node_api.h (tests/test_abi.py); the C-ABI
// it calls is tested from Python in tests/.
//
// Threading.  zkr.h requires the calls on one zkr_ctx to be serialised, and a zkr_pkey carries the work buffers of
// ONE proof in flight.  JS is free to overlap calls (two `await zkr.prove(...)` from concurrent Express requests,
// Promise.all, the tx and the withdraw generator together; a synchronous verify on the main thread while a prove
// runs on a libuv worker), so every zkr_* call on g_ctx below takes g_mu: proofs run one at a time per process,
// in the order the workers get the lock, and a key cannot be freed (GC finalizer) under a running proof.  One GPU
// holds one proof at a time anyway (the five-stream proof saturates it, DESIGN.md 4.4); to use several GPUs run one
// process per GPU or call zkr_prove_batch.
// Build (on a machine with node >= 12 and libzkr.so):
//   g++ -O2 -fPIC -shared -I$(node -p "require('node-addon-api').include_dir" || echo .) \
//       -I<node>/include/node -I../../include zkr_napi.cc -o zkr_napi.node -L.. -lzkr -Wl,-rpath,'$ORIGIN/..'
//
// Exposes to JS:
//   loadKey(pkBin: ArrayBuffer) -> keyHandle (external)            zkr_pkey_load_bin, once per circuit
//   loadKeyJson(pkJsonText: Buffer) -> keyHandle                   zkr_pkey_load_json: proving_key.json text, native parse
//   prove(key, witnessBin: ArrayBuffer, r?: Uint8Array(32), s?: Uint8Array(32)) -> Promise<Uint8Array(256)>
//        zkr_prove on a worker thread (napi_create_async_work), so the Express event loop never blocks
//        (the reference's websnark call is async for the same reason, operator/src/snarks/common.ts:29)
//   loadVerifyingKey(vkJsonText: Buffer) -> vkHandle               zkr_vkey_load_json, once per circuit
//   verify(vk, proof: Uint8Array(256), publicSignalsBin: ArrayBuffer) -> boolean
//        zkr_verify: replaces groth.isValid (common.ts:30-34); ~ms, synchronous
//   proveMany(key, witnessesBin: ArrayBuffer, rs?: Uint8Array(64 k)) -> Promise<Uint8Array(256 k)>
//        zkr_prove_many: k witnesses of the key back to back (k x nVars x 32 B), proved in one pass on a worker thread,
//        under the same mutex as prove; proof j is bytes [256 j, 256 (j+1)).  rs: k (r|s) pairs, or absent = CSPRNG.
//        The key's batch workspace (zkr_many) is created on first use, grown to the largest batch seen and freed with
//        the key.  common.ts's proveMany(key, witnesses[], rs?) -> Promise<Uint8Array[]> wraps it.
#include <node_api.h>

#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "zkr.h"

namespace {

zkr_ctx* g_ctx = nullptr;
std::mutex g_mu;             // serialises every zkr_* call on g_ctx (see "Threading" above)
using Lock = std::lock_guard<std::mutex>;
struct Many {
    zkr_many* mw = nullptr;
    int cap = 0;
};
std::map<zkr_pkey*, Many> g_many;          // proveMany's workspace per key, grown to the largest batch seen (under g_mu)

bool ensure_ctx(napi_env env) {
    Lock lk(g_mu);
    if (g_ctx) return true;
    int rc = zkr_ctx_create(0, &g_ctx);
    if (rc != ZKR_OK) {
        napi_throw_error(env, "ZKR_NO_DEVICE", zkr_last_error());   // no CPU fallback
        return false;
    }
    return true;
}

void free_key(napi_env, void* data, void*) {
    Lock lk(g_mu);
    zkr_pkey* pk = static_cast<zkr_pkey*>(data);
    zkr_many_free(g_many[pk].mw);        // proveMany's workspace shares the key's tables: freed first (null: none)
    g_many.erase(pk);
    zkr_pkey_free(pk);
}

napi_value LoadKey(napi_env env, napi_callback_info info) {
    size_t argc = 1;
    napi_value argv[1];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void* buf;
    size_t len;
    if (argc < 1 || napi_get_arraybuffer_info(env, argv[0], &buf, &len) != napi_ok) {
        napi_throw_type_error(env, nullptr, "loadKey(pkBin: ArrayBuffer)");
        return nullptr;
    }
    if (!ensure_ctx(env)) return nullptr;
    zkr_pkey* pk = nullptr;
    int rc;
    {
        Lock lk(g_mu);
        rc = zkr_pkey_load_bin(g_ctx, buf, len, &pk);
    }
    if (rc != ZKR_OK) {
        napi_throw_error(env, "ZKR_BADKEY", zkr_last_error());
        return nullptr;
    }
    napi_value ext;
    napi_create_external(env, pk, free_key, nullptr, &ext);
    return ext;
}

napi_value LoadKeyJson(napi_env env, napi_callback_info info) {
    size_t argc = 1;
    napi_value argv[1];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void* buf;
    size_t len;
    if (argc < 1 || napi_get_buffer_info(env, argv[0], &buf, &len) != napi_ok) {
        napi_throw_type_error(env, nullptr, "loadKeyJson(pkJsonText: Buffer)");
        return nullptr;
    }
    if (!ensure_ctx(env)) return nullptr;
    zkr_pkey* pk = nullptr;
    int rc;
    {
        Lock lk(g_mu);
        rc = zkr_pkey_load_json(g_ctx, static_cast<const char*>(buf), len, &pk);
    }
    if (rc != ZKR_OK) {
        napi_throw_error(env, "ZKR_BADKEY", zkr_last_error());
        return nullptr;
    }
    napi_value ext;
    napi_create_external(env, pk, free_key, nullptr, &ext);
    return ext;
}

void free_vkey(napi_env, void* data, void*) {
    Lock lk(g_mu);
    zkr_vkey_free(static_cast<zkr_vkey*>(data));
}

napi_value LoadVerifyingKey(napi_env env, napi_callback_info info) {
    size_t argc = 1;
    napi_value argv[1];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void* buf;
    size_t len;
    if (argc < 1 || napi_get_buffer_info(env, argv[0], &buf, &len) != napi_ok) {
        napi_throw_type_error(env, nullptr, "loadVerifyingKey(vkJsonText: Buffer)");
        return nullptr;
    }
    if (!ensure_ctx(env)) return nullptr;
    zkr_vkey* vk = nullptr;
    int rc;
    {
        Lock lk(g_mu);
        rc = zkr_vkey_load_json(g_ctx, static_cast<const char*>(buf), len, &vk);
    }
    if (rc != ZKR_OK) {
        napi_throw_error(env, "ZKR_BADKEY", zkr_last_error());
        return nullptr;
    }
    napi_value ext;
    napi_create_external(env, vk, free_vkey, nullptr, &ext);
    return ext;
}

// verify(vk, proof: Uint8Array(256), publicSignalsBin: ArrayBuffer of n x 32 B LE) -> boolean
napi_value Verify(napi_env env, napi_callback_info info) {
    size_t argc = 3;
    napi_value argv[3];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void *vkv, *pdata, *sbuf;
    size_t plen, slen, off;
    napi_typedarray_type ty;
    napi_value ab;
    if (argc < 3 || napi_get_value_external(env, argv[0], &vkv) != napi_ok ||
        napi_get_typedarray_info(env, argv[1], &ty, &plen, &pdata, &ab, &off) != napi_ok || plen != ZKR_PROOF_BYTES ||
        napi_get_arraybuffer_info(env, argv[2], &sbuf, &slen) != napi_ok || slen % 32) {
        napi_throw_type_error(env, nullptr, "verify(vk, proof: Uint8Array(256), publicSignalsBin: ArrayBuffer)");
        return nullptr;
    }
    int valid = 0, rc;
    {
        Lock lk(g_mu);       // waits for a proof in flight on a worker thread: the ctx's scratch and stream are shared
        rc = zkr_verify(g_ctx, static_cast<zkr_vkey*>(vkv), pdata, sbuf, slen / 32, &valid);
    }
    if (rc != ZKR_OK) {
        napi_throw_error(env, "ZKR_VERIFY", zkr_last_error());      // the contract's reverts (TxVerifier.sol:261,265)
        return nullptr;
    }
    napi_value out;
    napi_get_boolean(env, valid != 0, &out);
    return out;
}

struct ProveJob {
    napi_async_work work;
    napi_deferred deferred;
    zkr_pkey* pk;
    std::vector<uint8_t> witness;
    uint8_t r[32], s[32], proof[ZKR_PROOF_BYTES];
    bool has_r, has_s;
    int rc;
    std::string err;
};

void ProveExecute(napi_env, void* data) {       // worker thread
    ProveJob* j = static_cast<ProveJob*>(data);
    Lock lk(g_mu);
    // r / s absent: libzkr draws them from the OS CSPRNG (zkr.h), like websnark does internally
    j->rc = zkr_prove(g_ctx, j->pk, j->witness.data(), j->witness.size() / 32, j->has_r ? j->r : nullptr,
                      j->has_s ? j->s : nullptr, j->proof, nullptr);
    if (j->rc != ZKR_OK) j->err = zkr_last_error();      // thread-local message: read it on this thread
}

void ProveComplete(napi_env env, napi_status, void* data) {
    ProveJob* j = static_cast<ProveJob*>(data);
    if (j->rc == ZKR_OK) {
        void* out;
        napi_value ab, u8;
        napi_create_arraybuffer(env, ZKR_PROOF_BYTES, &out, &ab);
        memcpy(out, j->proof, ZKR_PROOF_BYTES);
        napi_create_typedarray(env, napi_uint8_array, ZKR_PROOF_BYTES, ab, 0, &u8);
        napi_resolve_deferred(env, j->deferred, u8);
    } else {
        napi_value msg, err;
        napi_create_string_utf8(env, j->err.c_str(), NAPI_AUTO_LENGTH, &msg);
        napi_create_error(env, nullptr, msg, &err);
        napi_reject_deferred(env, j->deferred, err);
    }
    napi_delete_async_work(env, j->work);
    delete j;
}

bool read_scalar(napi_env env, napi_value v, uint8_t out[32]) {
    napi_valuetype t;
    napi_typeof(env, v, &t);
    if (t == napi_undefined || t == napi_null) return false;
    napi_typedarray_type ty;
    size_t len;
    void* data;
    napi_value ab;
    size_t off;
    if (napi_get_typedarray_info(env, v, &ty, &len, &data, &ab, &off) != napi_ok || len != 32) return false;
    memcpy(out, data, 32);
    return true;
}

napi_value Prove(napi_env env, napi_callback_info info) {
    size_t argc = 4;
    napi_value argv[4];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void *pkv, *wbuf;
    size_t wlen;
    if (argc < 2 || napi_get_value_external(env, argv[0], &pkv) != napi_ok ||
        napi_get_arraybuffer_info(env, argv[1], &wbuf, &wlen) != napi_ok) {
        napi_throw_type_error(env, nullptr, "prove(key, witnessBin: ArrayBuffer, r?, s?)");
        return nullptr;
    }
    ProveJob* j = new ProveJob();
    j->pk = static_cast<zkr_pkey*>(pkv);
    j->witness.assign(static_cast<uint8_t*>(wbuf), static_cast<uint8_t*>(wbuf) + wlen);   // JS may GC the buffer
    j->has_r = argc > 2 && read_scalar(env, argv[2], j->r);
    j->has_s = argc > 3 && read_scalar(env, argv[3], j->s);
    napi_value promise, name;
    napi_create_promise(env, &j->deferred, &promise);
    napi_create_string_utf8(env, "zkr_prove", NAPI_AUTO_LENGTH, &name);
    napi_create_async_work(env, nullptr, name, ProveExecute, ProveComplete, j, &j->work);
    napi_queue_async_work(env, j->work);
    return promise;
}

struct ProveManyJob {
    napi_async_work work;
    napi_deferred deferred;
    zkr_pkey* pk;
    std::vector<uint8_t> witnesses, rs, proofs;
    int rc;
    std::string err;
    // whole witnesses of n_vars signals in the buffer (and as many (r|s) pairs, if given); 0 and rc set otherwise
    int count(uint32_t n_vars) {
        const size_t wb = 32ull * n_vars, k = wb ? witnesses.size() / wb : 0;
        if (k == 0 || k > 32767 || witnesses.size() != k * wb || (!rs.empty() && rs.size() != 64 * k)) {
            rc = ZKR_E_INVALID;
            err = "proveMany: witnessesBin must hold 1 .. 32767 whole witnesses of the key, rs one (r|s) pair per witness";
            return 0;
        }
        proofs.resize(ZKR_PROOF_BYTES * k);
        return (int)k;
    }
};

void ProveManyExecute(napi_env, void* data) {   // worker thread
    ProveManyJob* j = static_cast<ProveManyJob*>(data);
    Lock lk(g_mu);
    uint32_t n = 0;
    Many& m = g_many[j->pk];
    j->rc = zkr_pkey_info(j->pk, &n, nullptr, nullptr, nullptr);
    const int k = j->rc == ZKR_OK ? j->count(n) : 0;
    if (k > m.cap) zkr_many_free(m.mw), m = Many{}, j->rc = zkr_many_create(g_ctx, j->pk, k, &m.mw), m.cap = j->rc ? 0 : k;
    if (k > 0 && j->rc == ZKR_OK) j->rc = zkr_prove_many(g_ctx, m.mw, j->witnesses.data(), n, k, j->rs.empty() ? nullptr : j->rs.data(), j->proofs.data());
    if (j->rc != ZKR_OK && j->err.empty()) j->err = zkr_last_error();
}

void ProveManyComplete(napi_env env, napi_status, void* data) {
    ProveManyJob* j = static_cast<ProveManyJob*>(data);
    if (j->rc == ZKR_OK) {
        void* out;
        napi_value ab, u8;
        napi_create_arraybuffer(env, j->proofs.size(), &out, &ab);
        memcpy(out, j->proofs.data(), j->proofs.size());
        napi_create_typedarray(env, napi_uint8_array, j->proofs.size(), ab, 0, &u8);
        napi_resolve_deferred(env, j->deferred, u8);
    } else {
        napi_value msg, err;
        napi_create_string_utf8(env, j->err.c_str(), NAPI_AUTO_LENGTH, &msg);
        napi_create_error(env, nullptr, msg, &err);
        napi_reject_deferred(env, j->deferred, err);
    }
    napi_delete_async_work(env, j->work);
    delete j;
}

napi_value ProveMany(napi_env env, napi_callback_info info) {
    size_t argc = 3;
    napi_value argv[3];
    napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr);
    void *pkv, *wbuf, *rdata = nullptr;
    size_t wlen, rlen = 0;
    bool ok = argc >= 2 && napi_get_value_external(env, argv[0], &pkv) == napi_ok &&
              napi_get_arraybuffer_info(env, argv[1], &wbuf, &wlen) == napi_ok;
    if (ok && argc > 2) {
        napi_valuetype t;
        napi_typeof(env, argv[2], &t);
        if (t != napi_undefined && t != napi_null) {
            napi_typedarray_type ty;
            napi_value ab;
            size_t off;
            ok = napi_get_typedarray_info(env, argv[2], &ty, &rlen, &rdata, &ab, &off) == napi_ok && ty == napi_uint8_array;
        }
    }
    if (!ok) {
        napi_throw_type_error(env, nullptr, "proveMany(key, witnessesBin: ArrayBuffer, rs?: Uint8Array)");
        return nullptr;
    }
    ProveManyJob* j = new ProveManyJob();
    j->pk = static_cast<zkr_pkey*>(pkv);
    j->witnesses.assign(static_cast<uint8_t*>(wbuf), static_cast<uint8_t*>(wbuf) + wlen);   // JS may GC the buffers
    if (rdata) j->rs.assign(static_cast<uint8_t*>(rdata), static_cast<uint8_t*>(rdata) + rlen);
    napi_value promise, name;
    napi_create_promise(env, &j->deferred, &promise);
    napi_create_string_utf8(env, "zkr_prove_many", NAPI_AUTO_LENGTH, &name);
    napi_create_async_work(env, nullptr, name, ProveManyExecute, ProveManyComplete, j, &j->work);
    napi_queue_async_work(env, j->work);
    return promise;
}

napi_value Init(napi_env env, napi_value exports) {
    napi_value f;
    napi_create_function(env, "loadKey", NAPI_AUTO_LENGTH, LoadKey, nullptr, &f);
    napi_set_named_property(env, exports, "loadKey", f);
    napi_create_function(env, "prove", NAPI_AUTO_LENGTH, Prove, nullptr, &f);
    napi_set_named_property(env, exports, "prove", f);
    napi_create_function(env, "loadKeyJson", NAPI_AUTO_LENGTH, LoadKeyJson, nullptr, &f);
    napi_set_named_property(env, exports, "loadKeyJson", f);
    napi_create_function(env, "loadVerifyingKey", NAPI_AUTO_LENGTH, LoadVerifyingKey, nullptr, &f);
    napi_set_named_property(env, exports, "loadVerifyingKey", f);
    napi_create_function(env, "verify", NAPI_AUTO_LENGTH, Verify, nullptr, &f);
    napi_set_named_property(env, exports, "verify", f);
    napi_create_function(env, "proveMany", NAPI_AUTO_LENGTH, ProveMany, nullptr, &f);
    napi_set_named_property(env, exports, "proveMany", f);
    return exports;
}

}  // namespace

NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
