// crcnn_b200.hpp -- C++17 host side of the B200 engine: CrCNN's layer and network classes, same
// names, constructor parameter lists, public members and virtuals as the reference's
// CrCNN/src/*.h, implemented over the C ABI (include/crcnn_b200.h) instead of the process-global
// seal::Evaluator.  A CrCNN program switches by including this header instead of the reference's
// layer headers and adding `using namespace crcnn_b200;` (see INTEGRATION.md).
//
// Two type modes:
//   -DCRCNN_WITH_SEAL   Ciphertext / Plaintext / EvaluationKeys are SEAL 2.3.1's own classes
//                       (true drop-in; needs the SEAL headers and library at build time).
//   default             layout- and stream-compatible stand-ins (same in-memory word layout,
//                       same save()/load() byte format: SEAL/seal/ciphertext.cpp:103-130,
//                       plaintext.cpp:346-364), so the host logic builds and is tested where SEAL's
//                       sources are absent (the GPU box).
//
// Reference interfaces mirrored (file:line under /root/reference/CrCNN/src):
//   globals.h:10-16 (typedefs), layer.h:10-31, convolutionalLayer.h:33-45, fullyConnectedLayer.h:22-36,
//   poolingLayer.h:12-21, avgPoolingLayer.h:7-14, batchNormLayer.h:13-30, squareLayer.h:9-20,
//   network.h:11-39.
#pragma once
#include <chrono>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <functional>
#include <istream>
#include <map>
#include <memory>
#include <ostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/crcnn_b200.h"

#ifdef CRCNN_WITH_SEAL
#include "seal/seal.h"
#endif

namespace crcnn_b200 {

// ------------------------------------------------------------------------------------------------
// value types
// ------------------------------------------------------------------------------------------------
#ifdef CRCNN_WITH_SEAL
using seal::Ciphertext;
using seal::EvaluationKeys;
using seal::Plaintext;
#else
// Stand-in for seal::Plaintext: coeff_count words, values < t (NTT form: K*(n+1) words).
class Plaintext {
public:
    Plaintext() = default;
    explicit Plaintext(int coeff_count) : w_(coeff_count, 0) {}
    int coeff_count() const { return (int)w_.size(); }
    std::uint64_t *data() { return w_.data(); }
    const std::uint64_t *data() const { return w_.data(); }
    std::uint64_t &operator[](int i) { return w_[i]; }
    const std::uint64_t &operator[](int i) const { return w_[i]; }
    void resize(int coeff_count) { w_.resize(coeff_count, 0); }
    void save(std::ostream &s) const {
        std::int32_t c = coeff_count();
        s.write(reinterpret_cast<const char *>(&c), 4);
        s.write(reinterpret_cast<const char *>(w_.data()), (std::streamsize)w_.size() * 8);
    }
    void load(std::istream &s) {
        std::int32_t c = 0;
        s.read(reinterpret_cast<char *>(&c), 4);
        w_.assign(c, 0);
        s.read(reinterpret_cast<char *>(w_.data()), (std::streamsize)c * 8);
    }
private:
    std::vector<std::uint64_t> w_;
};

// Stand-in for seal::Ciphertext: uint64[size][K][n+1] plus the header fields SEAL serialises.
class Ciphertext {
public:
    Ciphertext() = default;
    Ciphertext(int size, int poly_coeff_count, int coeff_mod_count)
        : size_(size), pcc_(poly_coeff_count), cmc_(coeff_mod_count), w_((size_t)size * poly_coeff_count * coeff_mod_count, 0) {}
    int size() const { return size_; }
    int poly_coeff_count() const { return pcc_; }
    int coeff_mod_count() const { return cmc_; }
    std::uint64_t *data() { return w_.data(); }
    const std::uint64_t *data() const { return w_.data(); }
    std::uint64_t *data(int poly) { return w_.data() + (size_t)poly * pcc_ * cmc_; }
    std::uint64_t hash_block[4] = {0, 0, 0, 0};
    void save(std::ostream &s) const {
        s.write(reinterpret_cast<const char *>(hash_block), 32);
        std::int32_t h[3] = {size_, pcc_, cmc_};
        s.write(reinterpret_cast<const char *>(h), 12);
        s.write(reinterpret_cast<const char *>(w_.data()), (std::streamsize)w_.size() * 8);
    }
    void load(std::istream &s) {
        s.read(reinterpret_cast<char *>(hash_block), 32);
        std::int32_t h[3] = {0, 0, 0};
        s.read(reinterpret_cast<char *>(h), 12);
        size_ = h[0]; pcc_ = h[1]; cmc_ = h[2];
        w_.assign((size_t)size_ * pcc_ * cmc_, 0);
        s.read(reinterpret_cast<char *>(w_.data()), (std::streamsize)w_.size() * 8);
    }
private:
    int size_ = 0, pcc_ = 0, cmc_ = 0;
    std::vector<std::uint64_t> w_;
};
#endif

// CrCNN/src/globals.h:10-16
typedef std::vector<std::vector<std::vector<Ciphertext>>> ciphertext3D;
typedef std::vector<std::vector<std::vector<Plaintext>>> plaintext3D;
typedef std::vector<std::vector<Ciphertext>> ciphertext2D;
typedef std::vector<std::vector<Plaintext>> plaintext2D;
typedef std::vector<std::vector<std::vector<std::vector<Plaintext>>>> plaintext4D;
typedef std::vector<std::vector<std::vector<float>>> floatCube;

// ------------------------------------------------------------------------------------------------
// Runtime: replaces the process-global `Evaluator *evaluator` / `EvaluationKeys *ev_keys16`
// (CrCNN/src/globals.h:23,27).  One GPU context per process, like the reference's globals.
// ------------------------------------------------------------------------------------------------
class Runtime {
public:
    static Runtime &get() { static Runtime r; return r; }

    // setParameters (CrCNN/src/globals.cpp:25-56) as far as evaluation is concerned.
    void init(int n, const std::vector<std::uint64_t> &q, std::uint64_t t, int device = 0) {
        reset();
        int rc = crcnn_ctx_create(n, (int)q.size(), q.data(), t, device, &ctx_);
        if (rc) fail(rc, crcnn_last_error(nullptr));
        n_ = n; K_ = (int)q.size(); t_ = t;
    }
#ifdef CRCNN_WITH_SEAL
    // Derive (n, q, t) from the caller's SEALContext; remembers the EncryptionParameters so that
    // result ciphertexts carry the right parameter hash (SEAL/seal/ciphertext.h:119-123).
    void init(const seal::SEALContext &context, int device = 0) {
        std::vector<std::uint64_t> q;
        for (auto &m : context.coeff_modulus()) q.push_back(m.value());
        init(context.poly_modulus().coeff_count() - 1, q, context.plain_modulus().value(), device);
        parms_.reset(new seal::EncryptionParameters(context.parms()));
    }
    void setEvaluationKeys(const seal::EvaluationKeys &keys) {
        // (SEAL 2.3.1's const hash_block() accessors recurse into themselves -- ciphertext.h:612-615,
        //  evaluationkeys.h:163-166 -- so the non-const overload is used on purpose)
        if (!parms_ || const_cast<seal::EvaluationKeys &>(keys).hash_block() != parms_->hash_block())
            throw std::invalid_argument("evaluation_keys is not valid for encryption parameters");  // evaluator.cpp:899-902
        const auto &row = keys.data()[0];
        std::vector<int> sizes;
        std::vector<std::uint64_t> words;
        for (auto &ct : row) {
            sizes.push_back(ct.size());
            words.insert(words.end(), ct.data(), ct.data() + (size_t)ct.size() * K_ * (n_ + 1));
        }
        setEvaluationKeys(words.data(), sizes.data(), keys.decomposition_bit_count());
    }
    const seal::EncryptionParameters &parms() const { return *parms_; }
#endif
    void setEvaluationKeys(const std::uint64_t *words, const int *sizes, int dbc) {
        need();
        if (evk_) crcnn_evk_free(ctx_, evk_);
        evk_ = nullptr;
        check(crcnn_evk_upload(ctx_, words, dbc, sizes, &evk_));
    }
    void reset() {
        if (ctx_) {
            if (evk_) crcnn_evk_free(ctx_, evk_);
            crcnn_ctx_destroy(ctx_);
        }
        ctx_ = nullptr; evk_ = nullptr;
    }
    ~Runtime() { reset(); }

    crcnn_ctx *ctx() { need(); return ctx_; }
    crcnn_evk *evk() {
        if (!evk_) throw std::invalid_argument("not enough evaluation keys");  // evaluator.cpp:903-906
        return evk_;
    }
    int n() const { return n_; }
    int K() const { return K_; }
    std::uint64_t t() const { return t_; }
    size_t ct_words(int size = 2) const { return (size_t)size * K_ * (n_ + 1); }

    // C ABI status -> the exception type the reference's callers see from SEAL
    void check(int rc) { if (rc) fail(rc, crcnn_last_error(ctx_)); }

private:
    Runtime() = default;
    void need() { if (!ctx_) throw std::logic_error("crcnn_b200::Runtime::init() has not been called"); }
    [[noreturn]] static void fail(int rc, const char *msg) {
        if (rc == CRCNN_ERR_INVALID_ARGUMENT) throw std::invalid_argument(msg);
        throw std::runtime_error(std::string("crcnn_b200: ") + msg);
    }
    crcnn_ctx *ctx_ = nullptr;
    crcnn_evk *evk_ = nullptr;
    int n_ = 0, K_ = 0;
    std::uint64_t t_ = 0;
#ifdef CRCNN_WITH_SEAL
    std::unique_ptr<seal::EncryptionParameters> parms_;
#endif
};

// RAII handles over the C ABI objects
struct DeviceTensor {
    crcnn_tensor *t = nullptr;
    int zd = 0, xd = 0, yd = 0;
    int batch = 1;     // independent images stacked in front: device layout [batch][z][x][y] (the reference processes one image per call)
    bool owned = true; // false: a view of a tensor somebody else frees (the input buffers of a BatchServer)
    DeviceTensor() = default;
    DeviceTensor(crcnn_tensor *p, int z, int x, int y, int b = 1, bool own = true) : t(p), zd(z), xd(x), yd(y), batch(b), owned(own) {}
    DeviceTensor(DeviceTensor &&o) noexcept : t(o.t), zd(o.zd), xd(o.xd), yd(o.yd), batch(o.batch), owned(o.owned) { o.t = nullptr; }
    DeviceTensor &operator=(DeviceTensor &&o) noexcept {
        if (this != &o) { release(); t = o.t; zd = o.zd; xd = o.xd; yd = o.yd; batch = o.batch; owned = o.owned; o.t = nullptr; }
        return *this;
    }
    DeviceTensor(const DeviceTensor &) = delete;
    DeviceTensor &operator=(const DeviceTensor &) = delete;
    ~DeviceTensor() { release(); }
    void release() { if (t && owned) crcnn_tensor_free(Runtime::get().ctx(), t); t = nullptr; }
    long count() const { return (long)batch * zd * xd * yd; }
};

struct PlainPack {
    crcnn_plain *p = nullptr;
    PlainPack() = default;
    PlainPack(const PlainPack &) = delete;
    PlainPack &operator=(const PlainPack &) = delete;
    ~PlainPack() { clear(); }
    void clear() { if (p) crcnn_plain_free(Runtime::get().ctx(), p); p = nullptr; }
    // Coefficient-form plaintexts -> sparse device pack.  NTT-form plaintexts (coeff_count > n+1, what the
    // reference's layers leave behind after their first forward, convolutionalLayer.cpp:151-156) are rejected
    // like SEAL rejects them in transform_to_ntt (evaluator.cpp:1426-1429).
    void assign(const std::vector<const Plaintext *> &pts) {
        clear();
        Runtime &rt = Runtime::get();
        std::vector<std::uint32_t> off(1, 0), idx;
        std::vector<std::uint64_t> val;
        for (const Plaintext *pt : pts) {
            if (pt->coeff_count() > rt.n() + 1) throw std::invalid_argument("plain is not valid for encryption parameters");
            const std::uint64_t *w = pt->data();
            for (int c = 0; c < pt->coeff_count(); c++)
                if (w[c]) { idx.push_back((std::uint32_t)c); val.push_back(w[c]); }
            off.push_back((std::uint32_t)idx.size());
        }
        rt.check(crcnn_plain_upload_sparse(rt.ctx(), idx.data(), val.data(), off.data(), (long)pts.size(), &p));
    }
    // Floats -> FractionalEncoder(t, x^n+1, 64, 32, base 3) plaintexts on the device, as CnnBuilder encodes them
    // (CrCNN/src/cnnBuilder.cpp:25-105); no host Plaintext per weight (fc3 of PlainModel.h5 would be 41 GB of them).
    void encode(const std::vector<float> &values) {
        clear();
        Runtime &rt = Runtime::get();
        rt.check(crcnn_plain_encode(rt.ctx(), values.data(), (long)values.size(), &p));
    }
    // Host copy of plaintext `index` (coefficient form, n+1 words like the encoder's output)
    Plaintext fetch(long index) const {
        Runtime &rt = Runtime::get();
        Plaintext pt;
        pt.resize(rt.n() + 1);
        rt.check(crcnn_plain_get(rt.ctx(), p, index, pt.data()));
        return pt;
    }
};

// ciphertext3D <-> device
inline DeviceTensor upload(const ciphertext3D &in) {
    Runtime &rt = Runtime::get();
    const int zd = (int)in.size(), xd = (int)in[0].size(), yd = (int)in[0][0].size();
    const size_t w = rt.ct_words(2);
    std::vector<std::uint64_t> stage((size_t)zd * xd * yd * w);
    size_t i = 0;
    for (auto &plane : in)
        for (auto &row : plane)
            for (auto &ct : row) {
                if (ct.size() != 2 || ct.poly_coeff_count() != rt.n() + 1 || ct.coeff_mod_count() != rt.K())
                    throw std::invalid_argument("encrypted is not valid for encryption parameters");
#ifdef CRCNN_WITH_SEAL
                if (const_cast<Ciphertext &>(ct).hash_block() != rt.parms().hash_block())
                    throw std::invalid_argument("encrypted is not valid for encryption parameters");  // evaluator.cpp:1503-1506
#endif
                std::memcpy(stage.data() + i * w, ct.data(), w * 8);
                i++;
            }
    crcnn_tensor *t = nullptr;
    rt.check(crcnn_tensor_upload(rt.ctx(), stage.data(), (long)zd * xd * yd, 2, &t));
    rt.check(crcnn_ctx_sync(rt.ctx()));  // `stage` is pageable and about to go away
    return DeviceTensor(t, zd, xd, yd);
}

inline ciphertext3D download(const DeviceTensor &d) {
    Runtime &rt = Runtime::get();
    const size_t w = rt.ct_words(2);
    std::vector<std::uint64_t> stage((size_t)d.zd * d.xd * d.yd * w);
    rt.check(crcnn_tensor_download(rt.ctx(), d.t, stage.data()));
    ciphertext3D out(d.zd, ciphertext2D(d.xd, std::vector<Ciphertext>(d.yd)));
    size_t i = 0;
    for (auto &plane : out)
        for (auto &row : plane)
            for (auto &ct : row) {
#ifdef CRCNN_WITH_SEAL
                Ciphertext alias(rt.parms(), 2, stage.data() + i * w);  // sets the parameter hash
                ct = alias;                                              // deep copy, un-aliased
#else
                ct = Ciphertext(2, rt.n() + 1, rt.K());
                std::memcpy(ct.data(), stage.data() + i * w, w * 8);
#endif
                i++;
            }
    return out;
}

// ------------------------------------------------------------------------------------------------
// Encrypted-image files (CrCNN/src/globals.cpp:160-205): zd*xd*yd Ciphertext::save records back to back, [z][x][y] order.
// loadEncryptedImage / deepCopyImage keep the reference's signatures; saveEncryptedImage is the writing half of
// encryptAndSaveImage (the encryption itself stays with the key holder, SEAL on the host).
// ------------------------------------------------------------------------------------------------
inline ciphertext3D loadEncryptedImage(int zd, int xd, int yd, std::string file_name) {
    std::ifstream imagefile(file_name, std::ifstream::binary);
    if (!imagefile) throw std::invalid_argument("cannot open encrypted image " + file_name);
    ciphertext3D encrypted_image(zd, ciphertext2D(xd, std::vector<Ciphertext>(yd)));
    for (int z = 0; z < zd; z++)
        for (int i = 0; i < xd; i++)
            for (int j = 0; j < yd; j++) encrypted_image[z][i][j].load(imagefile);
    if (!imagefile) throw std::invalid_argument("encrypted image " + file_name + " is shorter than the requested shape");
    return encrypted_image;
}
inline void saveEncryptedImage(const ciphertext3D &encrypted_image, std::string file_name) {
    std::ofstream outfile(file_name, std::ofstream::binary);
    if (!outfile) throw std::invalid_argument("cannot write " + file_name);
    for (auto &plane : encrypted_image)
        for (auto &row : plane)
            for (auto &ct : row) ct.save(outfile);
}
inline ciphertext3D deepCopyImage(ciphertext3D image) { return image; }  // value semantics: the vectors copy every Ciphertext

// ------------------------------------------------------------------------------------------------
// Layer (CrCNN/src/layer.h:10-31)
// ------------------------------------------------------------------------------------------------
class Layer {
public:
    std::string name;
    Layer() {}
    Layer(std::string layer_name) : name(layer_name) {}
    virtual ~Layer() {}
    std::string getName() { return name; }
    virtual void printLayerStructure() = 0;
    // Reference signature: ciphertexts in and out by value on the host.
    virtual ciphertext3D forward(ciphertext3D input) { return download(forward_dev(upload(input))); }
    // Device-resident variant used by Network::forward so activations never leave HBM between layers.
    virtual DeviceTensor forward_dev(DeviceTensor input) = 0;
    virtual void savePlaintextParameters(std::ostream *outfile) = 0;
    virtual void loadPlaintextParameters(std::istream *infile) = 0;
    // CrCNN/src/layer.cpp:12-26
    void computeBoundaries(int xd, int yd, int xs, int ys, int xf, int yf, int *xl, int *yl) {
        *xl = (xf > xs) ? xd - xf + 1 : xd - xs + 1;
        *yl = (yf > ys) ? yd - yf + 1 : yd - ys + 1;
    }
};

// ------------------------------------------------------------------------------------------------
// ConvolutionalLayer (CrCNN/src/convolutionalLayer.h:9-58)
// ------------------------------------------------------------------------------------------------
class PoolingLayer;      // declared here so that member signatures below name THESE classes, not same-named ones of an including program
class BatchNormLayer;
class ConvolutionalLayer : public Layer {
public:
    int xd, yd, zd, xs, ys, xf, yf, nf, th_count;  // th_count is accepted and ignored (the GPU schedules the work)
    int xp, yp;   // zero padding: xp columns and yp rows of all-zero ciphertexts on each side of the input (0 in the reference's layers)
    int xo, yo, zo;
    plaintext4D filters;  // nf,zd,xf,yf -- never modified by forward (the reference NTT-transforms them in place)
    std::vector<Plaintext> biases;
    bool filters_already_ntt;  // kept for source compatibility; always false here

    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int th_count,
                       plaintext4D &filters, std::vector<Plaintext> &biases)
        : ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, 0, 0, th_count, filters, biases) {}
    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int th_count,
                       std::istream *infile)
        : ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, 0, 0, th_count, infile) {}
    // Trained floats in the reference's order [nf][zd][xf][yf] (cnnBuilder.cpp:36-47), encoded on the device; the host
    // members `filters` / `biases` stay empty until materializeHostParameters() (getKernel, getBias and save call it).
    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int th_count,
                       const std::vector<float> &weights, const std::vector<float> &bias_values)
        : ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, 0, 0, th_count, weights, bias_values) {}

    // The same three forms with zero padding (xp, yp), 0 <= xp < xf and 0 <= yp < yf: the layer computes what the reference's
    // forward computes on the input with a border of all-zero ciphertexts (crcnn_conv_forward_padded), and its output is
    // (xd + 2 xp - xf) / xs + 1 by (yd + 2 yp - yf) / ys + 1.  Padding is geometry: the parameter stream format is unchanged.
    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int xp, int yp, int th_count,
                       plaintext4D &filters, std::vector<Plaintext> &biases)
        : Layer(name), xd(xd), yd(yd), zd(zd), xs(xs), ys(ys), xf(xf), yf(yf), nf(nf), th_count(th_count), xp(checked_pad(xp, xf)),
          yp(checked_pad(yp, yf)), xo((xd + 2 * xp - xf) / xs + 1), yo((yd + 2 * yp - yf) / ys + 1), zo(nf), filters(filters), biases(biases),
          filters_already_ntt(false) {}
    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int xp, int yp, int th_count,
                       std::istream *infile)
        : Layer(name), xd(xd), yd(yd), zd(zd), xs(xs), ys(ys), xf(xf), yf(yf), nf(nf), th_count(th_count), xp(checked_pad(xp, xf)),
          yp(checked_pad(yp, yf)), xo((xd + 2 * xp - xf) / xs + 1), yo((yd + 2 * yp - yf) / ys + 1), zo(nf), filters_already_ntt(false) {
        loadPlaintextParameters(infile);
    }
    ConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int xp, int yp, int th_count,
                       const std::vector<float> &weights, const std::vector<float> &bias_values)
        : Layer(name), xd(xd), yd(yd), zd(zd), xs(xs), ys(ys), xf(xf), yf(yf), nf(nf), th_count(th_count), xp(checked_pad(xp, xf)),
          yp(checked_pad(yp, yf)), xo((xd + 2 * xp - xf) / xs + 1), yo((yd + 2 * yp - yf) / ys + 1), zo(nf), filters_already_ntt(false) {
        if ((long)weights.size() != (long)nf * zd * xf * yf || (int)bias_values.size() != nf) throw std::invalid_argument("kernel shape does not match the layer");
        w_.encode(weights); b_.encode(bias_values);
    }
    void materializeHostParameters() {
        if (!filters.empty() || !w_.p) return;
        filters.assign(nf, plaintext3D(zd, plaintext2D(xf, std::vector<Plaintext>(yf))));
        biases.resize(nf);
        long w = 0;
        for (int n = 0; n < nf; n++) {
            for (int z = 0; z < zd; z++)
                for (int i = 0; i < xf; i++)
                    for (int j = 0; j < yf; j++) filters[n][z][i][j] = w_.fetch(w++);
            biases[n] = b_.fetch(n);
        }
    }

    DeviceTensor forward_dev(DeviceTensor in) override {
        Runtime &rt = Runtime::get();
        ensure_packs();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_conv_forward_padded(rt.ctx(), in.t, w_.p, b_.p, in.batch, xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, 0, nf, &o));
        return DeviceTensor(o, zo, xo, yo, in.batch);
    }
    // Output channels [k0, k0+kc) only: this GPU's share of the reference's filter split (convolutionalLayer.cpp:177-187)
    DeviceTensor forward_shard(const DeviceTensor &in, int k0, int kc) {
        Runtime &rt = Runtime::get();
        ensure_packs();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_conv_forward_padded(rt.ctx(), in.t, w_.p, b_.p, in.batch, xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, k0, kc, &o));
        return DeviceTensor(o, kc, xo, yo, in.batch);
    }
    crcnn_plain *weight_pack() { ensure_packs(); return w_.p; }
    crcnn_plain *bias_pack() { ensure_packs(); return b_.p; }
    plaintext3D getKernel(int kernel_index) { materializeHostParameters(); return filters[kernel_index]; }
    Plaintext getBias(int bias_index) { materializeHostParameters(); return biases[bias_index]; }

    // stream format: per filter zd*xf*yf weight records then the bias (convolutionalLayer.cpp:213-229)
    void savePlaintextParameters(std::ostream *outfile) override {
        materializeHostParameters();
        for (int n = 0; n < nf; n++) {
            for (int z = 0; z < zd; z++)
                for (int i = 0; i < xf; i++)
                    for (int j = 0; j < yf; j++) { filters[n][z][i][j].save(*outfile); outfile->flush(); }
            biases[n].save(*outfile);
            outfile->flush();
        }
    }
    void loadPlaintextParameters(std::istream *infile) override {
        plaintext4D w(nf, plaintext3D(zd, plaintext2D(xf, std::vector<Plaintext>(yf))));
        std::vector<Plaintext> b(nf);
        for (int n = 0; n < nf; n++) {
            for (int z = 0; z < zd; z++)
                for (int i = 0; i < xf; i++)
                    for (int j = 0; j < yf; j++) w[n][z][i][j].load(*infile);
            b[n].load(*infile);
        }
        filters = w; biases = b;
        w_.clear(); b_.clear();
    }
    void printLayerStructure() override {
        std::fprintf(stderr, "Convolutional %s : input (%d,%d,%d); kernel(%d,%d,%d,%d); stride(%d,%d); padding(%d,%d); output(%d,%d,%d)\n",
                     name.c_str(), zd, xd, yd, nf, zd, xf, yf, xs, ys, xp, yp, zo, xo, yo);
    }

private:
    static int checked_pad(int pad, int filter) {
        if (pad < 0 || pad >= filter) throw std::invalid_argument("convolution padding must be in [0, filter - 1]");
        return pad;
    }
    void ensure_packs() {
        if (w_.p) return;
        std::vector<const Plaintext *> ws, bs;
        for (auto &f : filters) for (auto &pl : f) for (auto &row : pl) for (auto &p : row) ws.push_back(&p);
        for (auto &p : biases) bs.push_back(&p);
        if ((int)ws.size() != nf * zd * xf * yf || (int)bs.size() != nf) throw std::invalid_argument("kernel shape does not match the layer");
        w_.assign(ws); b_.assign(bs);
    }
    PlainPack w_, b_;
};

// ------------------------------------------------------------------------------------------------
// FullyConnectedLayer (CrCNN/src/fullyConnectedLayer.h:13-50)
// ------------------------------------------------------------------------------------------------
class FullyConnectedLayer : public Layer {
public:
    int in_dim, out_dim, th_count;
    plaintext2D weights;
    std::vector<Plaintext> biases;
    bool weights_already_ntt;

    FullyConnectedLayer(std::string name, int in_dim, int out_dim, int th_count, plaintext2D &weights, std::vector<Plaintext> &biases)
        : Layer(name), in_dim(in_dim), out_dim(out_dim), th_count(th_count), weights(weights), biases(biases), weights_already_ntt(false) {}
    FullyConnectedLayer(std::string name, int in_dim, int out_dim, int th_count, std::istream *infile)
        : Layer(name), in_dim(in_dim), out_dim(out_dim), th_count(th_count), weights_already_ntt(false) {
        loadPlaintextParameters(infile);
    }

    // Trained floats in the reference's order [out_dim][in_dim] (cnnBuilder.cpp:64-73), encoded on the device; `weights` /
    // `biases` stay empty until materializeHostParameters().
    FullyConnectedLayer(std::string name, int in_dim, int out_dim, int th_count, const std::vector<float> &weight_values,
                        const std::vector<float> &bias_values)
        : Layer(name), in_dim(in_dim), out_dim(out_dim), th_count(th_count), weights_already_ntt(false) {
        if ((long)weight_values.size() != (long)in_dim * out_dim || (int)bias_values.size() != out_dim) throw std::invalid_argument("weight shape does not match the layer");
        w_.encode(weight_values); b_.encode(bias_values);
    }
    void materializeHostParameters() {
        if (!weights.empty() || !w_.p) return;
        weights.assign(out_dim, std::vector<Plaintext>(in_dim));
        biases.resize(out_dim);
        for (int i = 0; i < out_dim; i++) {
            for (int j = 0; j < in_dim; j++) weights[i][j] = w_.fetch((long)i * in_dim + j);
            biases[i] = b_.fetch(i);
        }
    }

    // reshapeInput (fullyConnectedLayer.cpp:38-56): [z][x][y] -> [1][z*x*y][1], row-major.
    ciphertext3D reshapeInput(ciphertext3D input) {
        int x_size = (int)input[0].size(), y_size = (int)input[0][0].size(), z_size = (int)input.size();
        if (z_size != 1 && y_size != 1) {
            ciphertext3D r(1, ciphertext2D(in_dim, std::vector<Ciphertext>(1)));
            for (int i = 0; i < in_dim; ++i) {
                int z = i / (x_size * y_size), x = i / y_size - (x_size * z), y = i % y_size;
                r[0][i][0] = input[z][x][y];
            }
            return r;
        }
        return input;
    }
    DeviceTensor forward_dev(DeviceTensor in) override {
        Runtime &rt = Runtime::get();
        ensure_packs();
        // the device layout [z][x][y] is already the row-major flattening reshapeInput produces
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_fc_forward(rt.ctx(), in.t, w_.p, b_.p, in.batch, in_dim, out_dim, &o));
        return DeviceTensor(o, 1, out_dim, 1, in.batch);
    }
    // this layer and the fully connected layer that follows it directly, as one composed layer (crcnn_fc_fc_forward): what
    // Network::forward_dev calls for fc3 -> fc4 (cnnBuilder.cpp:121-122); the composed weights are built at the first call
    DeviceTensor forward_then(DeviceTensor in, FullyConnectedLayer &next) {
        Runtime &rt = Runtime::get();
        ensure_packs(); next.ensure_packs();
        if (next.in_dim != out_dim) throw std::invalid_argument("fully connected layers do not chain");
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_fc_fc_forward(rt.ctx(), in.t, w_.p, b_.p, next.w_.p, next.b_.p, in.batch, in_dim, out_dim, next.out_dim, &o));
        return DeviceTensor(o, 1, next.out_dim, 1, in.batch);
    }
    // avg-pool + batch-norm + this layer + the next one (crcnn_pool_bn_fc_fc_forward): layers 5-8 of the nine-layer networks
    DeviceTensor forward_after_avgpool_bn_then(DeviceTensor in, PoolingLayer &pool, BatchNormLayer &bn, FullyConnectedLayer &next);
    // Output rows [o0, o0+oc) only: this GPU's share of the reference's row split (fullyConnectedLayer.cpp:148-158)
    DeviceTensor forward_shard(const DeviceTensor &in, int o0, int oc) {
        Runtime &rt = Runtime::get();
        ensure_packs();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_fc_forward_shard(rt.ctx(), in.t, w_.p, b_.p, in.batch, in_dim, out_dim, o0, oc, &o));
        return DeviceTensor(o, 1, oc, 1, in.batch);
    }
    Plaintext getWeight(int x_index, int y_index) { materializeHostParameters(); return weights[x_index][y_index]; }
    Plaintext getBias(int x_index) { materializeHostParameters(); return biases[x_index]; }

    // per output row in_dim weights then the bias (fullyConnectedLayer.cpp:198-208)
    void savePlaintextParameters(std::ostream *outfile) override {
        materializeHostParameters();
        for (int i = 0; i < out_dim; i++) {
            for (int j = 0; j < in_dim; j++) { weights[i][j].save(*outfile); outfile->flush(); }
            biases[i].save(*outfile);
            outfile->flush();
        }
    }
    void loadPlaintextParameters(std::istream *infile) override {
        std::vector<Plaintext> b(out_dim);
        plaintext2D w(out_dim, std::vector<Plaintext>(in_dim));
        for (int i = 0; i < out_dim; i++) {
            for (int j = 0; j < in_dim; j++) w[i][j].load(*infile);
            b[i].load(*infile);
        }
        weights = w; biases = b;
        w_.clear(); b_.clear();
    }
    void printLayerStructure() override { std::fprintf(stderr, "FullyConnected %s : (%d -> %d)\n", name.c_str(), in_dim, out_dim); }

private:
    void ensure_packs() {
        if (w_.p) return;
        std::vector<const Plaintext *> ws, bs;
        for (auto &row : weights) for (auto &p : row) ws.push_back(&p);
        for (auto &p : biases) bs.push_back(&p);
        if ((int)ws.size() != in_dim * out_dim || (int)bs.size() != out_dim) throw std::invalid_argument("weight shape does not match the layer");
        w_.assign(ws); b_.assign(bs);
    }
    PlainPack w_, b_;
};

// ------------------------------------------------------------------------------------------------
// PoolingLayer / AvgPoolingLayer (CrCNN/src/poolingLayer.h:9-34, avgPoolingLayer.h:5-16)
// ------------------------------------------------------------------------------------------------
class PoolingLayer : public Layer {
public:
    int xd, yd, xs, ys, xf, yf, xo, yo, zo;
    PoolingLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf)
        : Layer(name), xd(xd), yd(yd), xs(xs), ys(ys), xf(xf), yf(yf), xo((xd - xf) / xs + 1), yo((yd - yf) / ys + 1), zo(zd) {}
    DeviceTensor forward_dev(DeviceTensor in) override {
        Runtime &rt = Runtime::get();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_pool_forward(rt.ctx(), in.t, in.batch, xd, yd, in.zd, xs, ys, xf, yf, scale(), &o));   // in.zd: a channel shard pools its own channels
        return DeviceTensor(o, in.zd, xo, yo, in.batch);
    }
    void printLayerStructure() override {
        std::fprintf(stderr, "Pooling %s : input (%d,%d,%d); kernel(%d,%d); stride(%d,%d); output(%d,%d,%d)\n", name.c_str(), zo, xd, yd, xf, yf, xs, ys, zo, xo, yo);
    }
    void savePlaintextParameters(std::ostream *) override {}
    void loadPlaintextParameters(std::istream *) override {}
    crcnn_plain *scale_or_null() { return scale(); }     // the 1/(xf*yf) pack of an AvgPoolingLayer, nullptr for a plain window sum
protected:
    virtual crcnn_plain *scale() { return nullptr; }
};

class AvgPoolingLayer : public PoolingLayer {
public:
    Plaintext div_factor;  // encode(1/(xf*yf)), avgPoolingLayer.cpp:10-13
    AvgPoolingLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf)
        : PoolingLayer(name, xd, yd, zd, xs, ys, xf, yf) {
        Runtime &rt = Runtime::get();
        double v = 1. / (xf * yf);   // a double, as in the reference (avgPoolingLayer.cpp:12): 1/9 as a float has other base-3 digits
        rt.check(crcnn_plain_encode_f64(rt.ctx(), &v, 1, &pack_.p));
        div_factor = Plaintext(rt.n() + 1);
        rt.check(crcnn_plain_get(rt.ctx(), pack_.p, 0, div_factor.data()));
    }
    crcnn_plain *scale_pack() { return pack_.p; }
protected:
    crcnn_plain *scale() override { return pack_.p; }
private:
    PlainPack pack_;
};

// ------------------------------------------------------------------------------------------------
// BatchNormLayer (CrCNN/src/batchNormLayer.h:10-40) -- `var` holds 1/sqrt(var+1e-5) as in the reference
// ------------------------------------------------------------------------------------------------
class BatchNormLayer : public Layer {
public:
    int num_channels;
    std::vector<Plaintext> mean;
    std::vector<Plaintext> var;
    BatchNormLayer(std::string name, int num_channels, std::vector<Plaintext> &mean, std::vector<Plaintext> &var)
        : Layer(name), num_channels(num_channels), mean(mean), var(var) {}
    BatchNormLayer(std::string name, int num_channels, std::istream *infile) : Layer(name), num_channels(num_channels) {
        loadPlaintextParameters(infile);
    }
    // running mean and 1/sqrt(running_var + 1e-5) as floats (cnnBuilder.cpp:96-103), encoded on the device
    BatchNormLayer(std::string name, int num_channels, const std::vector<float> &mean_values, const std::vector<float> &invstd_values)
        : Layer(name), num_channels(num_channels) {
        if ((int)mean_values.size() != num_channels || (int)invstd_values.size() != num_channels) throw std::invalid_argument("statistics do not match the channel count");
        m_.encode(mean_values); v_.encode(invstd_values);
        mean_f_ = mean_values; invstd_f_ = invstd_values;
    }
    // Channels [k0, k0+kc) of a channel-sharded activation (batch-norm is per channel: no exchange, SURVEY 8(e))
    DeviceTensor forward_shard(const DeviceTensor &in, int k0, int kc) {
        Runtime &rt = Runtime::get();
        if (k0 < 0 || kc < 0 || k0 + kc > num_channels || in.zd != kc) throw std::invalid_argument("bad channel shard");
        if (!sm_.p || s0_ != k0 || sc_ != kc) {
            if (!mean_f_.empty()) {
                sm_.encode(std::vector<float>(mean_f_.begin() + k0, mean_f_.begin() + k0 + kc));
                sv_.encode(std::vector<float>(invstd_f_.begin() + k0, invstd_f_.begin() + k0 + kc));
            } else {
                std::vector<const Plaintext *> ms, vs;
                for (int i = k0; i < k0 + kc; i++) { ms.push_back(&mean[i]); vs.push_back(&var[i]); }
                sm_.assign(ms); sv_.assign(vs);
            }
            s0_ = k0; sc_ = kc;
        }
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_bn_forward(rt.ctx(), in.t, in.batch, kc, in.xd, in.yd, sm_.p, sv_.p, &o));
        return DeviceTensor(o, kc, in.xd, in.yd, in.batch);
    }
    void materializeHostParameters() {
        if (!mean.empty() || !m_.p) return;
        mean.resize(num_channels); var.resize(num_channels);
        for (int i = 0; i < num_channels; i++) { mean[i] = m_.fetch(i); var[i] = v_.fetch(i); }
    }
    crcnn_plain *mean_pack() { ensure_packs(); return m_.p; }
    crcnn_plain *invstd_pack() { ensure_packs(); return v_.p; }
    void ensure_packs() {
        if (m_.p) return;
        std::vector<const Plaintext *> ms, vs;
        for (auto &p : mean) ms.push_back(&p);
        for (auto &p : var) vs.push_back(&p);
        m_.assign(ms); v_.assign(vs);
    }
    // avg-pool + this batch-norm in one pass over NTT-form activations (crcnn_pool_bn_forward): what Network::forward_dev calls when an
    // AvgPoolingLayer is directly followed by a BatchNormLayer (layers 1+2 and 5+6 of the reference's nine-layer blocks, cnnBuilder.cpp:115-134)
    DeviceTensor forward_after_avgpool(DeviceTensor in, PoolingLayer &pool);
    // convolution + avg-pool + this batch-norm (crcnn_conv_pool_bn_forward): layers 0-2 of those blocks; a stride-1 convolution is then
    // evaluated on the pooled grid (window sums of its input, convolution at the pooling stride) -- same bytes, a quarter of the columns
    DeviceTensor forward_after_conv_avgpool(DeviceTensor in, ConvolutionalLayer &conv, PoolingLayer &pool);
    // output channels [k0, k0+kc) of the same (ShardedNetwork); returns false -- and leaves `in` alone -- where the engine has no pooled-grid
    // path for this geometry (the caller then runs the three layers one by one on its shard)
    bool forward_after_conv_avgpool_shard(const DeviceTensor &in, ConvolutionalLayer &conv, PoolingLayer &pool, int k0, int kc, DeviceTensor *out);
    DeviceTensor forward_dev(DeviceTensor in) override {
        Runtime &rt = Runtime::get();
        ensure_packs();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_bn_forward(rt.ctx(), in.t, in.batch, in.zd, in.xd, in.yd, m_.p, v_.p, &o));
        return DeviceTensor(o, in.zd, in.xd, in.yd, in.batch);
    }
    Plaintext getMean(int index) { materializeHostParameters(); return mean[index]; }
    Plaintext getVar(int index) { materializeHostParameters(); return var[index]; }
    // alternating mean / var records (batchNormLayer.cpp:42-48)
    void savePlaintextParameters(std::ostream *outfile) override {
        materializeHostParameters();
        for (int i = 0; i < num_channels; i++) { mean[i].save(*outfile); var[i].save(*outfile); outfile->flush(); }
    }
    void loadPlaintextParameters(std::istream *infile) override {
        std::vector<Plaintext> m(num_channels), v(num_channels);
        for (int i = 0; i < num_channels; i++) { m[i].load(*infile); v[i].load(*infile); }
        mean = m; var = v;
        m_.clear(); v_.clear();
    }
    void printLayerStructure() override { std::fprintf(stderr, "BatchNormLayer2D %s :num_channels %d\n", name.c_str(), num_channels); }
private:
    PlainPack m_, v_, sm_, sv_;
    std::vector<float> mean_f_, invstd_f_;
    int s0_ = -1, sc_ = -1;
};

inline DeviceTensor BatchNormLayer::forward_after_avgpool(DeviceTensor in, PoolingLayer &pool) {
    Runtime &rt = Runtime::get();
    ensure_packs();
    if (in.zd != num_channels) throw std::invalid_argument("channel count of the pooled tensor does not match the batch-norm layer");
    crcnn_tensor *o = nullptr;
    rt.check(crcnn_pool_bn_forward(rt.ctx(), in.t, in.batch, pool.xd, pool.yd, in.zd, pool.xs, pool.ys, pool.xf, pool.yf, pool.scale_or_null(), m_.p, v_.p, &o));
    return DeviceTensor(o, in.zd, pool.xo, pool.yo, in.batch);
}

inline DeviceTensor BatchNormLayer::forward_after_conv_avgpool(DeviceTensor in, ConvolutionalLayer &conv, PoolingLayer &pool) {
    Runtime &rt = Runtime::get();
    ensure_packs();
    if (conv.nf != num_channels || pool.xd != conv.xo || pool.yd != conv.yo)
        throw std::invalid_argument("convolution / pooling / batch-norm shapes do not chain");
    crcnn_tensor *o = nullptr;
    rt.check(crcnn_conv_pool_bn_forward_padded(rt.ctx(), in.t, conv.weight_pack(), conv.bias_pack(), in.batch, conv.xd, conv.yd, conv.zd, conv.xs,
                                               conv.ys, conv.xf, conv.yf, conv.nf, pool.xs, pool.ys, pool.xf, pool.yf, pool.scale_or_null(), m_.p,
                                               v_.p, conv.xp, conv.yp, 0, conv.nf, &o));
    return DeviceTensor(o, conv.nf, pool.xo, pool.yo, in.batch);
}

inline DeviceTensor FullyConnectedLayer::forward_after_avgpool_bn_then(DeviceTensor in, PoolingLayer &pool, BatchNormLayer &bn, FullyConnectedLayer &next) {
    Runtime &rt = Runtime::get();
    ensure_packs(); next.ensure_packs();
    if (next.in_dim != out_dim || bn.num_channels != in.zd || in.zd * pool.xo * pool.yo != in_dim)
        throw std::invalid_argument("pooling / batch-norm / fully connected shapes do not chain");
    crcnn_tensor *o = nullptr;
    rt.check(crcnn_pool_bn_fc_fc_forward(rt.ctx(), in.t, in.batch, pool.xd, pool.yd, in.zd, pool.xs, pool.ys, pool.xf, pool.yf, pool.scale_or_null(),
                                         bn.mean_pack(), bn.invstd_pack(), w_.p, b_.p, next.w_.p, next.b_.p, out_dim, next.out_dim, &o));
    return DeviceTensor(o, 1, next.out_dim, 1, in.batch);
}

inline bool BatchNormLayer::forward_after_conv_avgpool_shard(const DeviceTensor &in, ConvolutionalLayer &conv, PoolingLayer &pool, int k0, int kc,
                                                             DeviceTensor *out) {
    Runtime &rt = Runtime::get();
    ensure_packs();
    if (conv.nf != num_channels || pool.xd != conv.xo || pool.yd != conv.yo)
        throw std::invalid_argument("convolution / pooling / batch-norm shapes do not chain");
    crcnn_tensor *o = nullptr;
    const int rc = crcnn_conv_pool_bn_forward_padded(rt.ctx(), in.t, conv.weight_pack(), conv.bias_pack(), in.batch, conv.xd, conv.yd, conv.zd, conv.xs,
                                                     conv.ys, conv.xf, conv.yf, conv.nf, pool.xs, pool.ys, pool.xf, pool.yf, pool.scale_or_null(), m_.p,
                                                     v_.p, conv.xp, conv.yp, k0, kc, &o);
    if (rc == CRCNN_ERR_UNSUPPORTED) return false;
    rt.check(rc);
    *out = DeviceTensor(o, kc, pool.xo, pool.yo, in.batch);
    return true;
}

// ------------------------------------------------------------------------------------------------
// SquareLayer (CrCNN/src/squareLayer.h:6-28)
// ------------------------------------------------------------------------------------------------
class SquareLayer : public Layer {
public:
    int th_count;
    SquareLayer(std::string name, int th_count) : Layer(name), th_count(th_count) {}
    SquareLayer() : th_count(1) {}
    DeviceTensor forward_dev(DeviceTensor in) override {
        Runtime &rt = Runtime::get();
        crcnn_tensor *o = nullptr;
        rt.check(crcnn_square_forward(rt.ctx(), in.t, rt.evk(), &o));
        return DeviceTensor(o, in.zd, in.xd, in.yd, in.batch);
    }
    void printLayerStructure() override { std::fprintf(stderr, "SquareLayer %s\n", name.c_str()); }
    void savePlaintextParameters(std::ostream *) override {}
    void loadPlaintextParameters(std::istream *) override {}
};

// ------------------------------------------------------------------------------------------------
// Network (CrCNN/src/network.h:11-39, network.cpp:22-47)
// ------------------------------------------------------------------------------------------------
class OutOfBudgetException : public std::exception {
public:
    const int last_layer_computed;
    OutOfBudgetException(int last_layer_computed) : last_layer_computed(last_layer_computed),
        msg_("OutOfBudgetException at layer " + std::to_string(last_layer_computed)) {}
    const char *what() const throw() override { return msg_.c_str(); }
private:
    std::string msg_;
};

// Several images -> ONE device tensor [batch][z][x][y] (one pinned staging buffer, one H2D copy)
inline DeviceTensor upload_batch(const std::vector<ciphertext3D> &images) {
    Runtime &rt = Runtime::get();
    if (images.empty()) throw std::invalid_argument("empty batch");
    const int B = (int)images.size(), zd = (int)images[0].size(), xd = (int)images[0][0].size(), yd = (int)images[0][0][0].size();
    const size_t w = rt.ct_words(2), per = (size_t)zd * xd * yd;
    void *pin = nullptr;
    if (crcnn_pinned_alloc(B * per * w * 8, &pin)) throw std::runtime_error("crcnn_b200: cannot allocate pinned staging memory");
    std::uint64_t *stage = static_cast<std::uint64_t *>(pin);
    size_t i = 0;
    try {
        for (auto &in : images) {
            if ((int)in.size() != zd || (int)in[0].size() != xd || (int)in[0][0].size() != yd) throw std::invalid_argument("images of a batch must have one shape");
            for (auto &plane : in)
                for (auto &row : plane)
                    for (auto &ct : row) {
                        if (ct.size() != 2 || ct.poly_coeff_count() != rt.n() + 1 || ct.coeff_mod_count() != rt.K())
                            throw std::invalid_argument("encrypted is not valid for encryption parameters");
                        std::memcpy(stage + i * w, ct.data(), w * 8);
                        i++;
                    }
        }
        crcnn_tensor *t = nullptr;
        rt.check(crcnn_tensor_upload(rt.ctx(), stage, (long)(B * per), 2, &t));
        rt.check(crcnn_ctx_sync(rt.ctx()));
        crcnn_pinned_free(pin);
        return DeviceTensor(t, zd, xd, yd, B);
    } catch (...) { crcnn_pinned_free(pin); throw; }
}

inline std::vector<ciphertext3D> download_batch(const DeviceTensor &d) {
    Runtime &rt = Runtime::get();
    const size_t w = rt.ct_words(2), per = (size_t)d.zd * d.xd * d.yd;
    std::vector<std::uint64_t> stage((size_t)d.batch * per * w);
    rt.check(crcnn_tensor_download(rt.ctx(), d.t, stage.data()));
    std::vector<ciphertext3D> out(d.batch, ciphertext3D(d.zd, ciphertext2D(d.xd, std::vector<Ciphertext>(d.yd))));
    size_t i = 0;
    for (auto &img : out)
        for (auto &plane : img)
            for (auto &row : plane)
                for (auto &ct : row) {
#ifdef CRCNN_WITH_SEAL
                    Ciphertext alias(rt.parms(), 2, stage.data() + i * w);
                    ct = alias;
#else
                    ct = Ciphertext(2, rt.n() + 1, rt.K());
                    std::memcpy(ct.data(), stage.data() + i * w, w * 8);
#endif
                    i++;
                }
    return out;
}

class Network {
public:
    std::vector<std::shared_ptr<Layer>> layers;
    // The reference re-encrypts (decrypt + encrypt with the SECRET key) unconditionally before layer 6
    // (network.cpp:23,30-38).  That step belongs to the key holder: install it in `reencrypt`.  A network with more than
    // layer_before_reenc layers and NO callback does not silently skip it: forward() throws std::logic_error unless the caller
    // has opted out with skip_reencryption = true (at n = 8192 the nine-layer networks have the budget to run without it: 96 bits
    // left after PlainModel's last layer, DESIGN 4.4 -- but then outputs and noise budgets differ from a reference run, and the
    // caller should know).  reencrypt_below_budget (below) replaces the fixed point by the budget-driven policy.
    int layer_before_reenc = 6;
    std::function<ciphertext3D(ciphertext3D)> reencrypt;
    bool skip_reencryption = false;
    // The same step WITHOUT leaving the device (SURVEY 8(f) N4): decrypt -> decode -> float -> encode -> encrypt of every activation
    // ciphertext on the GPU (crcnn_reencrypt), for a key holder who runs the evaluator himself -- the reference's own situation
    // (its Network::forward holds the secret key in process globals).  Takes precedence over `reencrypt` when set.
    std::function<DeviceTensor(DeviceTensor)> reencrypt_dev;
    // The key holder's keys on the device (opt-in, like the reference's own in-process keys): secret_key_ntt = SecretKey::data()
    // (NTT form, [K][n+1] words), public_key_ntt = PublicKey::data() ([2][K][n+1], NTT form).  Uploaded once and kept here; they
    // give noise_budgets / min_noise_budget and the adaptive policy below.
    std::shared_ptr<crcnn_keys> device_keys;
    void use_device_keys(const std::uint64_t *secret_key_ntt, const std::uint64_t *public_key_ntt) {
        Runtime &rt = Runtime::get();
        crcnn_keys *k = nullptr;
        rt.check(crcnn_keys_upload(rt.ctx(), secret_key_ntt, public_key_ntt, &k));
        device_keys.reset(k, [](crcnn_keys *p) { crcnn_keys_free(Runtime::get().ctx(), p); });
    }
    // use_device_keys + reencrypt_dev from those keys; every call draws fresh randomness from (seed, call number).
    void use_device_reencryption(const std::uint64_t *secret_key_ntt, const std::uint64_t *public_key_ntt, std::uint64_t seed) {
        use_device_keys(secret_key_ntt, public_key_ntt);
        std::shared_ptr<crcnn_keys> keys = device_keys;
        auto calls = std::make_shared<std::uint64_t>(0);
        reencrypt_dev = [keys, seed, calls](DeviceTensor x) {
            Runtime &r = Runtime::get();
            crcnn_tensor *o = nullptr;
            r.check(crcnn_reencrypt(r.ctx(), keys.get(), x.t, seed + 0x9E3779B97F4A7C15ull * (*calls)++, 0.0, nullptr, &o, nullptr, nullptr));
            return DeviceTensor(o, x.zd, x.xd, x.yd, x.batch);
        };
    }
#ifdef CRCNN_WITH_SEAL
    void use_device_keys(const seal::SecretKey &sk, const seal::PublicKey &pk) { use_device_keys(sk.data().data(), pk.data().data()); }
    void use_device_reencryption(const seal::SecretKey &sk, const seal::PublicKey &pk, std::uint64_t seed) {
        use_device_reencryption(sk.data().data(), pk.data().data(), seed);
    }
#endif
    // Decryptor::invariant_noise_budget of every ciphertext of x (crcnn_noise_budget), and their minimum; need use_device_keys.
    std::vector<int> noise_budgets(const DeviceTensor &x) {
        std::vector<int> b((size_t)x.count());
        Runtime::get().check(crcnn_noise_budget(Runtime::get().ctx(), require_keys(), x.t, b.data(), nullptr));
        return b;
    }
    int min_noise_budget(const DeviceTensor &x) {
        int m = 0;
        Runtime::get().check(crcnn_noise_budget(Runtime::get().ctx(), require_keys(), x.t, nullptr, &m));
        return m;
    }
    // encryptImage / decryptImage (CrCNN/src/globals.cpp:127-142, 207-233) on the device with the installed keys; need use_device_keys.
    // encrypt_images_dev: images[b][z][x][y] -> one tensor [batch][z][x][y], the layout upload_batch produces (crcnn_encrypt_values).
    // Every call draws fresh randomness from (seed, call number), as reencrypt_dev does; do not hand the same seed to both.
    DeviceTensor encrypt_images_dev(const std::vector<floatCube> &images, std::uint64_t seed) {
        crcnn_keys *keys = require_keys();
        if (images.empty() || images[0].empty() || images[0][0].empty() || images[0][0][0].empty()) throw std::invalid_argument("empty batch");
        const int B = (int)images.size(), zd = (int)images[0].size(), xd = (int)images[0][0].size(), yd = (int)images[0][0][0].size();
        std::vector<float> v;
        v.reserve((size_t)B * zd * xd * yd);
        for (auto &img : images) {
            if ((int)img.size() != zd) throw std::invalid_argument("images of a batch must have one shape");
            for (auto &plane : img) {
                if ((int)plane.size() != xd) throw std::invalid_argument("images of a batch must have one shape");
                for (auto &row : plane) {
                    if ((int)row.size() != yd) throw std::invalid_argument("images of a batch must have one shape");
                    v.insert(v.end(), row.begin(), row.end());
                }
            }
        }
        Runtime &rt = Runtime::get();
        crcnn_tensor *t = nullptr;
        rt.check(crcnn_encrypt_values(rt.ctx(), keys, v.data(), (long)v.size(), seed + 0x9E3779B97F4A7C15ull * encrypt_calls_++, 0.0, nullptr, &t));
        return DeviceTensor(t, zd, xd, yd, B);
    }
    // x as x.count() / (zd*xd*yd) images of [zd][xd][yd] floats (crcnn_decrypt_values: only the floats leave the device).
    std::vector<floatCube> decrypt_images_dev(const DeviceTensor &x, int zd, int xd, int yd) {
        crcnn_keys *keys = require_keys();
        const long per = (long)zd * xd * yd;
        if (per <= 0 || x.count() % per) throw std::invalid_argument("tensor is not a whole number of images of that shape");
        std::vector<float> v((size_t)x.count());
        Runtime::get().check(crcnn_decrypt_values(Runtime::get().ctx(), keys, x.t, v.data()));
        return images_of(v, zd, xd, yd);
    }
    // v (a whole number of zd*xd*yd images, in order) as images [b][z][x][y]
    static std::vector<floatCube> images_of(const std::vector<float> &v, int zd, int xd, int yd) {
        const size_t per = (size_t)zd * xd * yd;
        std::vector<floatCube> out(v.size() / per, floatCube(zd, std::vector<std::vector<float>>(xd, std::vector<float>(yd))));
        size_t i = 0;
        for (auto &img : out)
            for (auto &plane : img)
                for (auto &row : plane)
                    for (auto &f : row) f = v[i++];
        return out;
    }
    // The reference program's encrypt -> forward -> decrypt (CrCNN/src/mainparams.cpp:84-111) for a batch, activations never leaving
    // the device: encrypt_images_dev, forward_batch's path (fusion, fixed or budget-driven re-encryption), decrypt_images_dev.
    std::vector<floatCube> predict(const std::vector<floatCube> &images, std::uint64_t seed) {
        DeviceTensor y = forward_batch_dev(encrypt_images_dev(images, seed));
        return decrypt_images_dev(y, y.zd, y.xd, y.yd);
    }

    // Budget-driven re-encryption, the reference's commented-out alternative to the fixed point (network.cpp:52-96): at a value
    // >= 0, forward / forward_batch run forward_dev_adaptive instead of re-encrypting before layer_before_reenc.  -1: off.
    int reencrypt_below_budget = -1;
    struct BudgetCheck { int layer; int min_budget; bool reencrypted; };
    std::vector<BudgetCheck> budget_log;   // the checks of the last forward_dev_adaptive, in order
    // The whole network with a noise-budget check after every call: after each layer, or after the last layer of a composed group
    // (DESIGN 4.5) -- with fusion on, a drop inside a group is seen at the group's end; the fuse_* switches off give the reference's
    // layer-by-layer placement.  At a check after layer i with minimum budget b over the tensor (a batch is re-encrypted whole):
    // b == 0 throws OutOfBudgetException(i) (the tensor may already decrypt wrongly; the last layer too); 0 < b <= threshold before
    // the last layer re-encrypts with reencrypt_dev, else the host callback `reencrypt`, else throws OutOfBudgetException(i).
    DeviceTensor forward_dev_adaptive(DeviceTensor x) {
        require_keys();
        const int L = (int)layers.size();
        budget_log.clear();
        for (int i = 0; i < L;) {
            const int end = i + group_at(i, L).second;
            x = forward_dev(std::move(x), i, end);
            const int j = end - 1, b = min_noise_budget(x);
            budget_log.push_back({j, b, false});
            if (b == 0) throw OutOfBudgetException(j);
            if (b <= reencrypt_below_budget && end < L) {
                if (reencrypt_dev) x = reencrypt_dev(std::move(x));
                else if (reencrypt) {
                    std::vector<ciphertext3D> mid = download_batch(x);
                    for (auto &m : mid) m = reencrypt(m);
                    x = upload_batch(mid);
                } else throw OutOfBudgetException(j);
                budget_log.back().reencrypted = true;
            }
            i = end;
        }
        return x;
    }

    Network() {}
    virtual ~Network() {}
    int getNumLayers() { return (int)layers.size(); }
    virtual std::shared_ptr<Layer> getLayer(int i) { return layers[i]; }
    std::vector<std::shared_ptr<Layer>> &getLayers() { return layers; }
    void printNetworkStructure() {
        for (size_t i = 0; i < layers.size(); i++) { std::fprintf(stderr, "(%zu) : ", i); layers[i]->printLayerStructure(); }
    }
    // The composed groups of DESIGN 4.5 that forward_dev runs as one call (same bytes as layer by layer)
    enum class Group {
        Single,        // one layer
        ConvPoolBn,    // ConvolutionalLayer + AvgPoolingLayer + BatchNormLayer: the convolution on the pooled grid (crcnn_conv_pool_bn_forward)
        ConvPool,      // ConvolutionalLayer + (Avg)PoolingLayer with no batch-norm behind it (the Tiny topology, cnnBuilder.cpp:157-169):
                       // the same pooled-grid layer with an identity batch-norm (mean 0, factor 1: C = the pooling scale, D = 0)
        PoolBnFcFc,    // AvgPoolingLayer + BatchNormLayer + two FullyConnectedLayers: window sums + one composed layer (crcnn_pool_bn_fc_fc_forward)
        FcFc,          // FullyConnectedLayer directly followed by FullyConnectedLayer: one composed layer (crcnn_fc_fc_forward)
        PoolBn         // AvgPoolingLayer directly followed by BatchNormLayer: one pass instead of two (crcnn_pool_bn_forward)
    };
    // The group forward_dev runs from layer i of the range [i, last), and its number of layers.  ConvPoolBn tests no geometry here:
    // BatchNormLayer::forward_after_conv_avgpool throws where the three shapes do not chain, so a mismatch is an error, never other
    // bytes.  ConvPool tests it because the layer-by-layer path is what a conv + pool pair that does not chain must get.
    std::pair<Group, int> group_at(int i, int last) {
        auto at = [&](int k) { return layers[i + k].get(); };
        if (fuse_conv_pool_bn && i + 2 < last && dynamic_cast<ConvolutionalLayer *>(at(0)) && dynamic_cast<PoolingLayer *>(at(1)) &&
            dynamic_cast<BatchNormLayer *>(at(2)))
            return {Group::ConvPoolBn, 3};
        if (fuse_conv_pool_bn && i + 1 < last) {
            auto *conv = dynamic_cast<ConvolutionalLayer *>(at(0));
            auto *pool = conv ? dynamic_cast<PoolingLayer *>(at(1)) : nullptr;
            if (pool && pool->xd == conv->xo && pool->yd == conv->yo) return {Group::ConvPool, 2};
        }
        if (fuse_fc_fc && fuse_pool_bn && i + 3 < last && dynamic_cast<PoolingLayer *>(at(0)) && dynamic_cast<BatchNormLayer *>(at(1)) &&
            dynamic_cast<FullyConnectedLayer *>(at(2)) && dynamic_cast<FullyConnectedLayer *>(at(3)))
            return {Group::PoolBnFcFc, 4};
        if (fuse_fc_fc && i + 1 < last && dynamic_cast<FullyConnectedLayer *>(at(0)) && dynamic_cast<FullyConnectedLayer *>(at(1)))
            return {Group::FcFc, 2};
        if (fuse_pool_bn && i + 1 < last && dynamic_cast<PoolingLayer *>(at(0)) && dynamic_cast<BatchNormLayer *>(at(1)))
            return {Group::PoolBn, 2};
        return {Group::Single, 1};
    }
    // Segment API (SURVEY 8(f) N2): layers [first, last) without leaving the device; any batch.
    virtual DeviceTensor forward_dev(DeviceTensor x, int first, int last) {
        if (first < 0 || last > (int)layers.size() || first > last) throw std::invalid_argument("bad layer range");
        for (int i = first; i < last;) {
            const std::pair<Group, int> g = group_at(i, last);
            auto at = [&](int k) { return layers[i + k].get(); };
            switch (g.first) {
            case Group::ConvPoolBn:
                x = static_cast<BatchNormLayer *>(at(2))->forward_after_conv_avgpool(std::move(x), *static_cast<ConvolutionalLayer *>(at(0)),
                                                                                      *static_cast<PoolingLayer *>(at(1)));
                break;
            case Group::ConvPool: {
                auto *conv = static_cast<ConvolutionalLayer *>(at(0));
                auto *pool = static_cast<PoolingLayer *>(at(1));
                IdentityBn &id = identity_bn(conv->nf);
                Runtime &rt = Runtime::get();
                crcnn_tensor *o = nullptr;
                rt.check(crcnn_conv_pool_bn_forward_padded(rt.ctx(), x.t, conv->weight_pack(), conv->bias_pack(), x.batch, conv->xd, conv->yd,
                                                           conv->zd, conv->xs, conv->ys, conv->xf, conv->yf, conv->nf, pool->xs, pool->ys, pool->xf,
                                                           pool->yf, pool->scale_or_null(), id.mean.p, id.invstd.p, conv->xp, conv->yp, 0, conv->nf, &o));
                x = DeviceTensor(o, conv->nf, pool->xo, pool->yo, x.batch);
                break;
            }
            case Group::PoolBnFcFc:
                x = static_cast<FullyConnectedLayer *>(at(2))->forward_after_avgpool_bn_then(std::move(x), *static_cast<PoolingLayer *>(at(0)),
                                                                                             *static_cast<BatchNormLayer *>(at(1)),
                                                                                             *static_cast<FullyConnectedLayer *>(at(3)));
                break;
            case Group::FcFc:
                x = static_cast<FullyConnectedLayer *>(at(0))->forward_then(std::move(x), *static_cast<FullyConnectedLayer *>(at(1)));
                break;
            case Group::PoolBn:
                x = static_cast<BatchNormLayer *>(at(1))->forward_after_avgpool(std::move(x), *static_cast<PoolingLayer *>(at(0)));
                break;
            case Group::Single:
                x = at(0)->forward_dev(std::move(x));
                break;
            }
            if (after_layer) for (int k = 0; k < g.second; k++) after_layer(i + k);
            i += g.second;
        }
        return x;
    }
    // mean 0 / factor 1 packs per channel count, for chains that have no batch-norm of their own
    struct IdentityBn { PlainPack mean, invstd; };
    IdentityBn &identity_bn(int channels) {
        auto &slot = identity_bn_[channels];
        if (!slot) {
            slot = std::make_shared<IdentityBn>();
            slot->mean.encode(std::vector<float>((size_t)channels, 0.f));
            slot->invstd.encode(std::vector<float>((size_t)channels, 1.f));
        }
        return *slot;
    }
    std::map<int, std::shared_ptr<IdentityBn>> identity_bn_;
    bool fuse_fc_fc = !(std::getenv("CRCNN_FC_FC") && std::atoi(std::getenv("CRCNN_FC_FC")) == 0);   // A/B switch, same bytes
    bool fuse_conv_pool_bn = !(std::getenv("CRCNN_CONV_POOL_BN") && std::atoi(std::getenv("CRCNN_CONV_POOL_BN")) == 0);   // A/B switch, same bytes
    bool fuse_pool_bn = !(std::getenv("CRCNN_POOL_BN") && std::atoi(std::getenv("CRCNN_POOL_BN")) == 0);   // A/B switch, same bytes
    // Called after layer i has been ENQUEUED (nothing has necessarily run yet): the place to record a CUDA event for per-layer timing,
    // the counterpart of the reference's commented-out chrono timers around layers[i]->forward (network.cpp:39-43).
    std::function<void(int)> after_layer;
    bool needs_reencryption() const { return layer_before_reenc > 0 && layer_before_reenc < (int)layers.size(); }
    crcnn_keys *require_keys() {
        if (!device_keys) throw std::logic_error("crcnn_b200::Network: noise budgets, encryption and decryption need the key holder's keys (use_device_keys)");
        return device_keys.get();
    }
    ciphertext3D forward(ciphertext3D input) {
        const int L = (int)layers.size();
        if (reencrypt_below_budget >= 0) return download(forward_dev_adaptive(upload(input)));
        if (needs_reencryption() && !skip_reencryption) {
            if (reencrypt_dev)
                return download(forward_dev(reencrypt_dev(forward_dev(upload(input), 0, layer_before_reenc)), layer_before_reenc, L));
            if (!reencrypt)
                throw std::logic_error("crcnn_b200::Network::forward: the reference re-encrypts before layer " + std::to_string(layer_before_reenc) +
                                       " (CrCNN/src/network.cpp:30); install Network::reencrypt (the key holder's decrypt + encrypt), call use_device_reencryption, or set skip_reencryption = true");
            ciphertext3D mid = download(forward_dev(upload(input), 0, layer_before_reenc));
            return download(forward_dev(upload(reencrypt(mid)), layer_before_reenc, L));
        }
        return download(forward_dev(upload(input), 0, L));
    }
    // Same for a batch of independent images in one pass (what the reference's per-image loop, mainparams.cpp:84-111, does one by one).
    std::vector<ciphertext3D> forward_batch(const std::vector<ciphertext3D> &inputs) { return download_batch(forward_batch_dev(upload_batch(inputs))); }
    // forward_batch's path on a device tensor [batch][z][x][y]
    DeviceTensor forward_batch_dev(DeviceTensor x) {
        const int L = (int)layers.size();
        if (reencrypt_below_budget >= 0) return forward_dev_adaptive(std::move(x));
        if (needs_reencryption() && !skip_reencryption) {
            if (reencrypt_dev) return forward_dev(reencrypt_dev(forward_dev(std::move(x), 0, layer_before_reenc)), layer_before_reenc, L);
            if (!reencrypt) throw std::logic_error("crcnn_b200::Network::forward_batch: re-encryption before layer " + std::to_string(layer_before_reenc) + " is not installed (see Network::forward)");
            std::vector<ciphertext3D> mid = download_batch(forward_dev(std::move(x), 0, layer_before_reenc));
            for (auto &m : mid) m = reencrypt(m);
            return forward_dev(upload_batch(mid), layer_before_reenc, L);
        }
        return forward_dev(std::move(x), 0, L);
    }
private:
    std::uint64_t encrypt_calls_ = 0;   // encrypt_images_dev's call number
};

// ------------------------------------------------------------------------------------------------
// BatchServer: the inference loop of the reference's program (CrCNN/src/mainparams.cpp:84-111: encrypt -> forward -> decrypt, one
// image at a time) as a double-buffered pipeline over batches.  Two device input tensors and one staging buffer are allocated
// once; while batch i runs on the context's stream, batch i+1 is copied host -> device on a copy stream
// (crcnn_tensor_upload_into) and the scores of batch i-1 are on their way back (crcnn_tensor_download_async).  Nothing is
// allocated per request and the host never blocks on the device except in wait().
// ------------------------------------------------------------------------------------------------
class BatchServer {
public:
    // zd, xd, yd: input shape of the network; batch: images per request; outputs: score ciphertexts per image
    BatchServer(Network &net, int zd, int xd, int yd, int batch, int outputs)
        : net_(net), zd_(zd), xd_(xd), yd_(yd), batch_(batch), outputs_(outputs) {
        Runtime &rt = Runtime::get();
        rt.check(crcnn_stream_create(rt.ctx(), &copy_));
        for (int i = 0; i < 2; i++) {
            rt.check(crcnn_tensor_wrap_alloc(rt.ctx(), (long)batch * zd * xd * yd, 2, 0, &in_[i]));
            rt.check(crcnn_event_create(rt.ctx(), &consumed_[i]));
            rt.check(crcnn_event_create(rt.ctx(), &done_[i]));
        }
    }
    ~BatchServer() {
        Runtime &rt = Runtime::get();
        crcnn_ctx_sync(rt.ctx());
        for (int i = 0; i < 2; i++) {
            if (in_[i]) crcnn_tensor_free(rt.ctx(), in_[i]);
            crcnn_event_destroy(rt.ctx(), consumed_[i]);
            crcnn_event_destroy(rt.ctx(), done_[i]);
        }
        crcnn_stream_destroy(rt.ctx(), copy_);
    }
    size_t input_words() const { return (size_t)batch_ * zd_ * xd_ * yd_ * Runtime::get().ct_words(2); }
    size_t output_words() const { return (size_t)batch_ * outputs_ * Runtime::get().ct_words(2); }

    // Stage request `seq` (0, 1, 2 ...): enqueue the upload of its input (pinned, SEAL layout, [batch][z][x][y]) on the copy stream.
    void stage(long seq, const std::uint64_t *pinned_in) {
        Runtime &rt = Runtime::get();
        const int slot = (int)(seq & 1);
        if (seq >= 2) rt.check(crcnn_stream_wait_event(rt.ctx(), copy_, consumed_[slot]));   // the forward that read this buffer has finished
        rt.check(crcnn_tensor_upload_into(rt.ctx(), pinned_in, in_[slot], 0, copy_));
    }
    // Run request `seq` (staged before) and enqueue the download of its scores into pinned_out; returns without waiting.
    void run(long seq, std::uint64_t *pinned_out) {
        Runtime &rt = Runtime::get();
        const int slot = (int)(seq & 1);
        rt.check(crcnn_ctx_wait_stream(rt.ctx(), copy_));
        DeviceTensor y = net_.forward_dev(DeviceTensor(in_[slot], zd_, xd_, yd_, batch_, /*own=*/false), 0, net_.getNumLayers());
        rt.check(crcnn_event_record(rt.ctx(), consumed_[slot], nullptr));
        if (y.count() != (long)batch_ * outputs_) throw std::logic_error("network output does not match BatchServer::outputs");
        rt.check(crcnn_tensor_download_async(rt.ctx(), y.t, pinned_out));
        rt.check(crcnn_event_record(rt.ctx(), done_[slot], nullptr));
    }
    // Block until the scores of request `seq` are in host memory.
    void wait(long seq) {
        Runtime &rt = Runtime::get();
        double ms;
        rt.check(crcnn_event_elapsed_ms(rt.ctx(), done_[seq & 1], done_[seq & 1], &ms));
    }
    // The whole loop for `requests` requests reading in(i) and writing out(i): upload of i+1 overlaps forward of i.
    void serve(long requests, const std::function<const std::uint64_t *(long)> &in, const std::function<std::uint64_t *(long)> &out) {
        if (requests <= 0) return;
        const auto t0 = std::chrono::steady_clock::now();
        auto stamp = [&] { completed_ms.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count()); };
        completed_ms.clear();
        stage(0, in(0));
        for (long i = 0; i < requests; i++) {
            run(i, out(i));                       // waits (on the device) for upload i, then forward + async score download
            if (i + 1 < requests) stage(i + 1, in(i + 1));
            if (i >= 1) { wait(i - 1); stamp(); } // scores of the previous request are complete: the caller may decrypt them
        }
        wait(requests - 1);
        stamp();
    }
    std::vector<double> completed_ms;   // host clock, from the start of the last serve(), at which each request's scores had landed
    void *copy_stream() { return copy_; }

private:
    Network &net_;
    int zd_, xd_, yd_, batch_, outputs_;
    void *copy_ = nullptr;
    crcnn_tensor *in_[2] = {nullptr, nullptr};
    void *consumed_[2] = {nullptr, nullptr}, *done_[2] = {nullptr, nullptr};
};

// ------------------------------------------------------------------------------------------------
// ShardedNetwork: one network split across the GPUs of a box by OUTPUT NEURON (SURVEY 8(e) item 3) -- the reference's own
// thread split (convolutionalLayer.cpp:177-187, fullyConnectedLayer.cpp:148-158) with GPUs in place of threads.  One process per
// GPU; every process holds the whole encoded network and calls forward_dev with the same input; conv / fc layers compute this
// rank's contiguous range of output channels / rows; pooling, batch-norm and square act on the local channels without any
// exchange; before a conv / fc layer (and at the end) the ranks all-gather their ciphertexts over NVLink (crcnn_comm_all_gather:
// one NCCL group on the context's stream, no host synchronisation).  Bit-identical to the unsharded forward.
// ------------------------------------------------------------------------------------------------
class ShardedNetwork : public Network {
public:
    ShardedNetwork(int world, int rank, const void *nccl_id128) : world_(world), rank_(rank) {
        Runtime &rt = Runtime::get();
        rt.check(crcnn_comm_create(rt.ctx(), nccl_id128, world, rank, &comm_));
    }
    ~ShardedNetwork() override { if (comm_) crcnn_comm_destroy(Runtime::get().ctx(), comm_); }
    int world() const { return world_; }
    int rank() const { return rank_; }
    // contiguous, balanced split: the first total % world ranks get one more (a rank may get none when world > total)
    static void shard_range(int total, int world, int rank, int *first, int *count) {
        const int base = total / world, extra = total % world;
        *first = rank * base + (rank < extra ? rank : extra);
        *count = base + (rank < extra ? 1 : 0);
    }
    DeviceTensor all_gather(const DeviceTensor &x, int channels, int per_channel, int xd, int yd) {
        Runtime &rt = Runtime::get();
        std::vector<long> counts(world_);
        for (int r = 0; r < world_; r++) { int f, c; shard_range(channels, world_, r, &f, &c); counts[r] = (long)c * per_channel; }
        crcnn_tensor *full = nullptr;
        rt.check(crcnn_comm_all_gather(rt.ctx(), comm_, x.t, x.batch, counts.data(), gather_ntt_form, &full));
        return DeviceTensor(full, channels, xd, yd, x.batch);
    }
    // x holds the FULL input on every rank; the result is the full output of layer last-1 on every rank.
    DeviceTensor forward_dev(DeviceTensor x, int first, int last) override {
        bool sharded = false;       // x holds only this rank's channels
        bool rows = false;          // ... which are output rows of a fully connected layer
        int channels = x.zd;
        for (int i = first; i < last; i++) {
            Layer *l = layers[i].get();
            if (auto *c = dynamic_cast<ConvolutionalLayer *>(l)) {
                if (sharded) x = all_gather(x, channels, x.xd * x.yd, x.xd, x.yd);
                int k0, kc; shard_range(c->nf, world_, rank_, &k0, &kc);
                // conv + pool + batch-norm: this rank's channels of the composed layer (§4.5 of DESIGN.md), when the engine has it for the geometry
                if (fuse_conv_pool_bn && i + 2 < last) {
                    auto *pool = dynamic_cast<PoolingLayer *>(layers[i + 1].get());
                    auto *bn = pool ? dynamic_cast<BatchNormLayer *>(layers[i + 2].get()) : nullptr;
                    DeviceTensor y;
                    if (bn && bn->forward_after_conv_avgpool_shard(x, *c, *pool, k0, kc, &y)) {
                        x = std::move(y);
                        channels = c->nf; sharded = true; rows = false;
                        if (after_layer) { after_layer(i); after_layer(i + 1); after_layer(i + 2); }
                        i += 2;
                        continue;
                    }
                }
                x = c->forward_shard(x, k0, kc);
                channels = c->nf; sharded = true; rows = false;
            } else if (auto *f = dynamic_cast<FullyConnectedLayer *>(l)) {
                if (sharded) x = all_gather(x, channels, x.xd * x.yd, x.xd, x.yd);
                // fc -> fc whose composed layer has only a handful of rows (fc3 * fc4: 10): every rank evaluates the composed layer on the gathered
                // input -- no split of fc3's rows, no second exchange
                auto *f2 = (fuse_fc_fc && i + 1 < last) ? dynamic_cast<FullyConnectedLayer *>(layers[i + 1].get()) : nullptr;
                if (f2 && f2->out_dim < min_sharded_outputs && (double)f2->out_dim * f->in_dim < (double)f->out_dim * (f->in_dim + f2->out_dim)) {
                    x = f->forward_then(std::move(x), *f2);
                    channels = 1; sharded = false; rows = false;
                    if (after_layer) { after_layer(i); after_layer(i + 1); }
                    i++;
                    continue;
                }
                if (f->out_dim < min_sharded_outputs) {
                    // a handful of output rows (fc4: 10): the layer's cost is transforming and staging its INPUT, which every rank has in
                    // full after the gather -- splitting the rows saves nothing and costs another exchange; every rank computes them all
                    x = f->forward_dev(std::move(x));
                    channels = 1; sharded = false; rows = false;
                } else {
                    int o0, oc; shard_range(f->out_dim, world_, rank_, &o0, &oc);
                    x = f->forward_shard(x, o0, oc);
                    x.zd = oc; x.xd = 1;            // rows play the part of channels for the next gather
                    channels = f->out_dim; sharded = true; rows = true;
                }
            } else if (auto *bn = dynamic_cast<BatchNormLayer *>(l)) {
                if (sharded) { int k0, kc; shard_range(channels, world_, rank_, &k0, &kc); x = bn->forward_shard(x, k0, kc); }
                else x = bn->forward_dev(std::move(x));
            } else {
                x = l->forward_dev(std::move(x));   // pooling and square are per channel / per ciphertext: local channels, no exchange
            }
            if (after_layer) after_layer(i);        // a layer's time includes the all-gather in front of it
        }
        if (sharded) {
            x = all_gather(x, channels, x.xd * x.yd, x.xd, x.yd);
            if (rows) { x.zd = 1; x.xd = channels; }   // a fully connected output is [1][out_dim][1] (fullyConnectedLayer.cpp:113-168)
        }
        return x;
    }
    int min_sharded_outputs = 32;   // fully connected layers with fewer output rows run replicated (no split, no exchange)
    int gather_ntt_form = -1;  // domain the activations are exchanged in: -1 as produced (no transform), 0 coefficient form, 1 NTT form

private:
    int world_, rank_;
    crcnn_comm *comm_ = nullptr;
};

// ------------------------------------------------------------------------------------------------
// CrtEnsemble: a large plain modulus T split into pairwise coprime t_1 .. t_M (BASELINE config 4), one independent instance of the
// network per GPU and process.  Each rank builds the whole network with CnnBuilder under Runtime::init(n, q, t_rank) and installs the
// key holder's keys (use_device_keys; the instances may share one key set: FV keys depend on n and q only).  The ensemble recombines
// the instances' plaintexts modulo T on the device (crcnn_crt_*), so the fixed re-encryption before layer_before_reenc and the final
// decryption see what one network under T sees, and predict returns on every rank the floats of a single Network::predict under T.
// The re-encryption and the decryption are collective: every rank must make the same calls in the same order.  That is why the
// budget-driven policy (reencrypt_below_budget >= 0) is refused -- each rank would decide from its own budget whether to re-encrypt.
// ------------------------------------------------------------------------------------------------
class CrtEnsemble {
public:
    // Collective (crcnn_crt_create).  Installs the collective re-encryption as net.reencrypt_dev; every call draws fresh randomness
    // from (reencrypt_seed, call number, rank).
    CrtEnsemble(Network &net, const std::vector<std::uint64_t> &moduli, int world, int rank, const void *nccl_id128, std::uint64_t reencrypt_seed)
        : net_(net) {
        net.require_keys();
        refuse_budget_policy();
        Runtime &rt = Runtime::get();
        rt.check(crcnn_comm_create(rt.ctx(), nccl_id128, world, rank, &comm_));
        try {
            rt.check(crcnn_crt_create(rt.ctx(), comm_, moduli.data(), (int)moduli.size(), &crt_));
        } catch (...) {
            crcnn_comm_destroy(rt.ctx(), comm_);
            throw;
        }
        Network *np = &net;
        crcnn_crt *crt = crt_;
        auto calls = std::make_shared<std::uint64_t>(0);
        net.reencrypt_dev = [np, crt, reencrypt_seed, calls](DeviceTensor x) {
            if (np->reencrypt_below_budget >= 0) throw std::logic_error(budget_policy_refused);
            Runtime &r = Runtime::get();
            crcnn_tensor *o = nullptr;
            r.check(crcnn_crt_reencrypt(r.ctx(), crt, np->require_keys(), x.t, reencrypt_seed + 0x9E3779B97F4A7C15ull * (*calls)++, 0.0, &o));
            return DeviceTensor(o, x.zd, x.xd, x.yd, x.batch);
        };
    }
    ~CrtEnsemble() {
        net_.reencrypt_dev = nullptr;
        crcnn_crt_free(Runtime::get().ctx(), crt_);
        crcnn_comm_destroy(Runtime::get().ctx(), comm_);
    }
    CrtEnsemble(const CrtEnsemble &) = delete;
    CrtEnsemble &operator=(const CrtEnsemble &) = delete;

    // Network::decrypt_images_dev under T (collective, crcnn_crt_decrypt_values): the same floats on every rank.
    std::vector<floatCube> decrypt_images_dev(const DeviceTensor &x, int zd, int xd, int yd) {
        crcnn_keys *keys = net_.require_keys();
        const long per = (long)zd * xd * yd;
        if (per <= 0 || x.count() % per) throw std::invalid_argument("tensor is not a whole number of images of that shape");
        std::vector<float> v((size_t)x.count());
        Runtime::get().check(crcnn_crt_decrypt_values(Runtime::get().ctx(), crt_, keys, x.t, v.data()));
        return Network::images_of(v, zd, xd, yd);
    }
    // Network::predict of the ensemble: this rank's instance encrypts the images (encrypt_images_dev) and runs forward_batch_dev,
    // re-encrypting collectively before layer_before_reenc; the scores are decrypted collectively.  Every rank calls it with the
    // same images and gets the same floats.
    std::vector<floatCube> predict(const std::vector<floatCube> &images, std::uint64_t seed) {
        refuse_budget_policy();
        DeviceTensor y = net_.forward_batch_dev(net_.encrypt_images_dev(images, seed));
        return decrypt_images_dev(y, y.zd, y.xd, y.yd);
    }

private:
    static constexpr const char *budget_policy_refused =
        "crcnn_b200::CrtEnsemble: the budget-driven re-encryption (reencrypt_below_budget >= 0) would let each rank decide alone whether "
        "to enter the collective re-encryption";
    void refuse_budget_policy() const { if (net_.reencrypt_below_budget >= 0) throw std::logic_error(budget_policy_refused); }
    Network &net_;
    crcnn_comm *comm_ = nullptr;
    crcnn_crt *crt_ = nullptr;
};

}  // namespace crcnn_b200
