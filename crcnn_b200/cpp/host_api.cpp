// host_api.cpp -- the C++17 host path (crcnn_b200.hpp: Runtime, CnnBuilder, Network, ShardedNetwork, BatchServer) behind a few
// extern "C" entry points, built into crcnn_b200/libcrcnn_b200_host.so.  bench.py and the GPU tests call THIS, so the numbers they
// report are produced by the same C++ code a CrCNN program links (the reference's inference program is C++:
// CrCNN/src/mainparams.cpp:64-116 builds the encoded network with CnnBuilder and loops images through Network::forward);
// Python stays the harness (rank plumbing, clocks, JSON).  One network per process, like the reference's globals.
#include <chrono>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "cnn_builder.hpp"

using namespace crcnn_b200;

namespace {
std::string g_err;
std::unique_ptr<Network> g_net;
std::unique_ptr<CrtEnsemble> g_crt;   // crcnn_host_crt_begin: this rank's place in a CRT ensemble over g_net
std::unique_ptr<BatchServer> g_srv;
std::unique_ptr<DeviceTensor> g_x0;   // resident input of crcnn_host_resident_*
int g_zd = 0, g_xd = 0, g_yd = 0, g_outputs = 0, g_batch = 0;

int g_oob_layer = -1;                 // layer of the last OutOfBudgetException

template <class F> int guarded(F &&f) {
    try { f(); return 0; }
    catch (const OutOfBudgetException &e) { g_err = e.what(); g_oob_layer = e.last_layer_computed; return CRCNN_ERR_OUT_OF_BUDGET; }
    catch (const std::invalid_argument &e) { g_err = e.what(); return CRCNN_ERR_INVALID_ARGUMENT; }
    catch (const std::exception &e) { g_err = e.what(); return CRCNN_ERR_CUDA; }
}
}  // namespace

extern "C" {

const char *crcnn_host_last_error() { return g_err.c_str(); }

// setParameters (CrCNN/src/globals.cpp:25-56) as far as evaluation goes
int crcnn_host_init(int n, int K, const uint64_t *q, uint64_t t, int device) {
    return guarded([&] { g_x0.reset(); g_srv.reset(); g_crt.reset(); g_net.reset(); Runtime::get().init(n, std::vector<uint64_t>(q, q + K), t, device); });
}
int crcnn_host_set_evk(const uint64_t *words, const int *sizes, int dbc) {
    return guarded([&] { Runtime::get().setEvaluationKeys(words, sizes, dbc); });
}
void *crcnn_host_ctx() { try { return Runtime::get().ctx(); } catch (...) { return nullptr; } }

// CnnBuilder(h5).buildNetwork(topology) (CrCNN/src/cnnBuilder.cpp:108-179).  world > 1: a ShardedNetwork over an NCCL communicator
// made from nccl_id (crcnn_comm_unique_id on rank 0, handed to every rank by the launcher).
int crcnn_host_build(const char *h5_path, const char *topology, int world, int rank, const void *nccl_id, int skip_reencryption) {
    return guarded([&] {
        g_x0.reset(); g_srv.reset(); g_crt.reset(); g_net.reset();
        CnnBuilder builder(h5_path);
        if (world > 1 || nccl_id) g_net.reset(new ShardedNetwork(world, rank, nccl_id));
        else g_net.reset(new Network());
        builder.buildLayers(*g_net, topology, "");
        g_net->skip_reencryption = skip_reencryption != 0;
        CnnBuilder::topologyShape(topology, &g_zd, &g_xd, &g_yd, &g_outputs);
    });
}
int crcnn_host_shape(int *zd, int *xd, int *yd, int *outputs, int *layers) {
    if (!g_net) { g_err = "no network built"; return CRCNN_ERR_INVALID_ARGUMENT; }
    *zd = g_zd; *xd = g_xd; *yd = g_yd; *outputs = g_outputs; *layers = g_net->getNumLayers();
    return 0;
}
int crcnn_host_layer_name(int i, char *name, int cap) {
    if (!g_net || i < 0 || i >= g_net->getNumLayers()) return CRCNN_ERR_INVALID_ARGUMENT;
    std::strncpy(name, g_net->getLayer(i)->name.c_str(), cap - 1);
    name[cap - 1] = 0;
    return 0;
}

// Layers [first, last) on `batch` images given as host words [batch][zd][xd][yd] ciphertexts (SEAL layout); the result's shape
// comes back in out_shape[3] and its ciphertexts in out_words (capacity out_cap words).  Segment API of SURVEY 8(f) N2.
int crcnn_host_forward_range(const uint64_t *in_words, int batch, int zd, int xd, int yd, int first, int last, uint64_t *out_words,
                             long out_cap, int *out_shape) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        Runtime &rt = Runtime::get();
        crcnn_tensor *t = nullptr;
        rt.check(crcnn_tensor_upload(rt.ctx(), in_words, (long)batch * zd * xd * yd, 2, &t));
        DeviceTensor y = g_net->forward_dev(DeviceTensor(t, zd, xd, yd, batch), first, last);
        if ((long)y.count() * (long)rt.ct_words(2) > out_cap) throw std::invalid_argument("output buffer too small");
        rt.check(crcnn_tensor_download(rt.ctx(), y.t, out_words));
        out_shape[0] = y.zd; out_shape[1] = y.xd; out_shape[2] = y.yd;
    });
}

// Forwards of the whole network with the input resident in HBM.  begin: upload the batch once and keep it; run: `steps` forwards,
// every one from a fresh coefficient-form copy of the resident input (so the input transform is inside the timed region), timed with
// CUDA events on the context's stream (ms_total) and per layer (per_layer_ms, mean over the steps; may be null); end: release.
// Warm-up and timed steps are separate run() calls on the SAME resident tensor, so the caller can put its barrier between them and the
// stream-ordered allocator sees one steady allocation pattern.  last_out (may be null): host words [batch][outputs] ciphertexts that
// receive the output of the last step, downloaded after the timing has ended.
int crcnn_host_resident_begin(const uint64_t *pinned_in, int batch) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        Runtime &rt = Runtime::get();
        crcnn_tensor *x0 = nullptr;
        rt.check(crcnn_tensor_upload(rt.ctx(), pinned_in, (long)batch * g_zd * g_xd * g_yd, 2, &x0));
        g_x0.reset(new DeviceTensor(x0, g_zd, g_xd, g_yd, batch));
    });
}
int crcnn_host_resident_run(int steps, double *ms_total, double *per_layer_ms, uint64_t *last_out) {
    return guarded([&] {
        if (!g_net || !g_x0) throw std::invalid_argument("crcnn_host_resident_begin has not been called");
        Runtime &rt = Runtime::get();
        crcnn_ctx *ctx = rt.ctx();
        const long count = g_x0->count();
        const int L = g_net->getNumLayers();
        std::vector<void *> ev((size_t)steps * (L + 1), nullptr);
        for (auto &e : ev) rt.check(crcnn_event_create(ctx, &e));
        DeviceTensor last;
        for (int s = 0; s < steps; s++) {
            crcnn_tensor *c = nullptr;
            rt.check(crcnn_tensor_slice(ctx, g_x0->t, 0, count, &c));
            DeviceTensor x(c, g_zd, g_xd, g_yd, g_x0->batch);
            rt.check(crcnn_event_record(ctx, ev[(size_t)s * (L + 1)], nullptr));
            // ONE pass over the whole network (a sharded network keeps its activations sharded between layers); an event after every layer.
            // The final all-gather of a sharded network lands after the last layer's event: one more event closes the step.
            g_net->after_layer = [&](int i) { rt.check(crcnn_event_record(ctx, ev[(size_t)s * (L + 1) + i + 1], nullptr)); };
            x = g_net->forward_dev(std::move(x), 0, L);
            g_net->after_layer = nullptr;
            rt.check(crcnn_event_record(ctx, ev[(size_t)s * (L + 1) + L], nullptr));
            if (last_out && s == steps - 1) last = std::move(x);
        }
        if (steps > 0 && ms_total) rt.check(crcnn_event_elapsed_ms(ctx, ev[0], ev[(size_t)(steps - 1) * (L + 1) + L], ms_total));
        if (per_layer_ms)
            for (int i = 0; i < L; i++) {
                double acc = 0;
                for (int s = 0; s < steps; s++) { double ms; rt.check(crcnn_event_elapsed_ms(ctx, ev[(size_t)s * (L + 1) + i], ev[(size_t)s * (L + 1) + i + 1], &ms)); acc += ms; }
                per_layer_ms[i] = steps ? acc / steps : 0;
            }
        rt.check(crcnn_ctx_sync(ctx));
        for (auto &e : ev) crcnn_event_destroy(ctx, e);
        if (last.t) {
            if (last.count() != (long)g_x0->batch * g_outputs) throw std::logic_error("network output is not [batch][outputs] ciphertexts");
            rt.check(crcnn_tensor_download(ctx, last.t, last_out));
        }
    });
}
int crcnn_host_resident_end() { return guarded([&] { g_x0.reset(); }); }

// The serving loop (BatchServer): `requests` requests of `batch` images, every one uploaded from pinned_in (host, SEAL layout)
// and its scores downloaded into pinned_out, upload of request i+1 overlapping the forward of request i.  ms_total = device time
// between an event before the first upload and the arrival of the last scores.
int crcnn_host_serve(const uint64_t *pinned_in, uint64_t *pinned_out, int batch, long requests, double *ms_total) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        Runtime &rt = Runtime::get();
        crcnn_ctx *ctx = rt.ctx();
        if (!g_srv || g_batch != batch) { g_srv.reset(new BatchServer(*g_net, g_zd, g_xd, g_yd, batch, g_outputs)); g_batch = batch; }
        void *e0 = nullptr, *e1 = nullptr;
        rt.check(crcnn_event_create(ctx, &e0));
        rt.check(crcnn_event_create(ctx, &e1));
        rt.check(crcnn_event_record(ctx, e0, nullptr));
        rt.check(crcnn_stream_wait_event(ctx, g_srv->copy_stream(), e0));     // the first upload starts inside the timed region
        g_srv->serve(requests, [&](long) { return pinned_in; }, [&](long) { return pinned_out; });
        rt.check(crcnn_event_record(ctx, e1, nullptr));
        rt.check(crcnn_event_elapsed_ms(ctx, e0, e1, ms_total));
        crcnn_event_destroy(ctx, e0); crcnn_event_destroy(ctx, e1);
    });
}

// Layer fusion of the built network on (default) / off: off runs every reference layer as its own call (A/B timing; same bytes).
int crcnn_host_set_fusion(int on) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        g_net->fuse_fc_fc = g_net->fuse_conv_pool_bn = g_net->fuse_pool_bn = on != 0;
    });
}

// The key holder's keys for the built network (Network::use_device_keys; with device_reencryption, use_device_reencryption with
// `seed`): secret_key_ntt [K][n+1], public_key_ntt [2][K][n+1] words, NTT form, as SEAL keeps them.
int crcnn_host_use_keys(const uint64_t *secret_key_ntt, const uint64_t *public_key_ntt, int device_reencryption, uint64_t seed) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        if (!secret_key_ntt || !public_key_ntt) throw std::invalid_argument("null key");
        g_net->reencrypt_dev = nullptr;
        if (device_reencryption) g_net->use_device_reencryption(secret_key_ntt, public_key_ntt, seed);
        else g_net->use_device_keys(secret_key_ntt, public_key_ntt);
    });
}
// Network::reencrypt_below_budget (-1: the fixed re-encryption point; >= 0: budget-driven re-encryption)
int crcnn_host_set_budget_threshold(int threshold) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        g_net->reencrypt_below_budget = threshold;
    });
}
// Network::forward_dev_adaptive on `batch` images given as host words [batch][zd][xd][yd] ciphertexts; output as in
// crcnn_host_forward_range.  An OutOfBudgetException returns CRCNN_ERR_OUT_OF_BUDGET with its layer in *failed_layer (may be null).
int crcnn_host_forward_adaptive(const uint64_t *in_words, int batch, uint64_t *out_words, long out_cap, int *out_shape, int *failed_layer) {
    g_oob_layer = -1;
    const int rc = guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        Runtime &rt = Runtime::get();
        crcnn_tensor *t = nullptr;
        rt.check(crcnn_tensor_upload(rt.ctx(), in_words, (long)batch * g_zd * g_xd * g_yd, 2, &t));
        DeviceTensor y = g_net->forward_dev_adaptive(DeviceTensor(t, g_zd, g_xd, g_yd, batch));
        if ((long)y.count() * (long)rt.ct_words(2) > out_cap) throw std::invalid_argument("output buffer too small");
        rt.check(crcnn_tensor_download(rt.ctx(), y.t, out_words));
        out_shape[0] = y.zd; out_shape[1] = y.xd; out_shape[2] = y.yd;
    });
    if (failed_layer) *failed_layer = g_oob_layer;
    return rc;
}
// Network::predict on `batch` images given as floats [batch][zd][xd][yd] (the built network's input shape): encrypted on the device
// with the installed keys (use_keys) from `seed` and the call number, forward_batch's path, decrypted on the device into
// scores[batch][outputs].  An OutOfBudgetException returns CRCNN_ERR_OUT_OF_BUDGET with its layer in *failed_layer (may be null).
int crcnn_host_predict_values(const float *images, int batch, uint64_t seed, float *scores, int *failed_layer) {
    g_oob_layer = -1;
    const int rc = guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        if (!images || !scores || batch <= 0) throw std::invalid_argument("bad predict arguments");
        std::vector<floatCube> in((size_t)batch, floatCube(g_zd, std::vector<std::vector<float>>(g_xd, std::vector<float>(g_yd))));
        const float *p = images;
        for (auto &img : in)
            for (auto &plane : img)
                for (auto &row : plane)
                    for (auto &f : row) f = *p++;
        const std::vector<floatCube> out = g_net->predict(in, seed);
        size_t i = 0;
        for (auto &img : out) {
            long per = 0;
            for (auto &plane : img)
                for (auto &row : plane) per += (long)row.size();
            if (per != g_outputs) throw std::logic_error("network output is not [batch][outputs] values");
            for (auto &plane : img)
                for (auto &row : plane)
                    for (float f : row) scores[i++] = f;
        }
    });
    if (failed_layer) *failed_layer = g_oob_layer;
    return rc;
}
// Network::budget_log of the last adaptive forward: (layer, minimum budget, re-encrypted) per check; returns how many there are.
int crcnn_host_budget_log(int *layer, int *min_budget, int *reencrypted, int cap) {
    if (!g_net) return 0;
    const int n = (int)g_net->budget_log.size();
    for (int i = 0; i < n && i < cap; i++) {
        layer[i] = g_net->budget_log[i].layer;
        min_budget[i] = g_net->budget_log[i].min_budget;
        reencrypted[i] = g_net->budget_log[i].reencrypted ? 1 : 0;
    }
    return n;
}

// Host-clock completion time (ms since the start of the last crcnn_host_serve) of each of its requests; returns how many there are.
int crcnn_host_serve_times(double *out, int cap) {
    if (!g_srv) return 0;
    const int n = (int)g_srv->completed_ms.size();
    for (int i = 0; i < n && i < cap; i++) out[i] = g_srv->completed_ms[i];
    return n;
}

// CrtEnsemble over the built network (after crcnn_host_build with world 1 and crcnn_host_use_keys): this rank holds the instance under
// moduli[rank] (the plain modulus of crcnn_host_init); collective, every rank of the M calls it with the same list and nccl_id.
// reencrypt_seed keys the noise of the collective re-encryption before layer 6.
int crcnn_host_crt_begin(const uint64_t *moduli, int M, int rank, const void *nccl_id, uint64_t reencrypt_seed) {
    return guarded([&] {
        if (!g_net) throw std::invalid_argument("no network built");
        if (!moduli || M < 1 || !nccl_id) throw std::invalid_argument("bad ensemble arguments");
        g_crt.reset();
        g_crt.reset(new CrtEnsemble(*g_net, std::vector<uint64_t>(moduli, moduli + M), M, rank, nccl_id, reencrypt_seed));
    });
}
// CrtEnsemble::predict, images and scores as in crcnn_host_predict_values; the same scores on every rank.
int crcnn_host_crt_predict_values(const float *images, int batch, uint64_t seed, float *scores) {
    return guarded([&] {
        if (!g_crt) throw std::invalid_argument("crcnn_host_crt_begin has not been called");
        if (!images || !scores || batch <= 0) throw std::invalid_argument("bad predict arguments");
        std::vector<floatCube> in((size_t)batch, floatCube(g_zd, std::vector<std::vector<float>>(g_xd, std::vector<float>(g_yd))));
        const float *p = images;
        for (auto &img : in)
            for (auto &plane : img)
                for (auto &row : plane)
                    for (auto &f : row) f = *p++;
        const std::vector<floatCube> out = g_crt->predict(in, seed);
        size_t i = 0;
        for (auto &img : out)
            for (auto &plane : img)
                for (auto &row : plane)
                    for (float f : row) {
                        if (i == (size_t)batch * g_outputs) throw std::logic_error("network output is not [batch][outputs] values");
                        scores[i++] = f;
                    }
        if (i != (size_t)batch * g_outputs) throw std::logic_error("network output is not [batch][outputs] values");
    });
}

void crcnn_host_shutdown() { g_x0.reset(); g_srv.reset(); g_crt.reset(); g_net.reset(); Runtime::get().reset(); }

}  // extern "C"
