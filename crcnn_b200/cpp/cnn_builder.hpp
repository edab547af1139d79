// cnn_builder.hpp -- CnnBuilder of the reference (CrCNN/src/cnnBuilder.h:16-52, cnnBuilder.cpp:9-196) over the B200 engine:
// reads the trained floats from a PlainModel*.h5 file (h5lite.hpp instead of libhdf5), encodes them with the reference's
// FractionalEncoder parameters ON THE DEVICE (crcnn_plain_encode) and assembles the encoded network out of the drop-in
// layer classes of crcnn_b200.hpp.  Same member names and argument lists as the reference; what differs:
//   * build*Layer with infile == NULL hands the floats to the layer's float constructor -- no host Plaintext per weight
//     (the reference materialises nf*zd*xf*yf + in*out seal::Plaintexts: 41 GB for fc3 of PlainModel.h5 at n = 8192);
//     the host members are filled on demand (materializeHostParameters) when a caller asks for them or saves the net;
//   * buildNetwork(file_name) builds the reference's ACTIVE block (PlainModelTiny, cnnBuilder.cpp:157-169);
//     buildNetwork(topology, file_name) also offers the two blocks the reference keeps commented out (Approx, WoPad,
//     cnnBuilder.cpp:115-155), "PlainModelPadded" = the weights file PlainModel.h5 as it was trained, conv1 with padding 2 on a
//     28x28 input, and "PlainModel" = the same weights run on a 32x32 input that carries the zero border itself
//     (SURVEY.md 8(a): that file has no builder block in the reference, whose layers have no padding).
// The simulator builders (buildSimulatedNetwork, ChooserPoly) are out of scope: noise estimation, not the forward path.
#pragma once
#include <cmath>
#include <fstream>

#include "crcnn_b200.hpp"
#include "h5lite.hpp"

namespace crcnn_b200 {

class CnnBuilder {
public:
    std::string plain_model_path;
    LoadH5 ldata;

    CnnBuilder(std::string plain_model_path) : plain_model_path(plain_model_path) { ldata.setFileName(plain_model_path); }
    ~CnnBuilder() {}

    // cnnBuilder.cpp:20-23
    std::vector<float> getPretrained(std::string var_name) {
        ldata.setVarName(var_name);
        return ldata.getData();
    }

    // cnnBuilder.cpp:25-51
    ConvolutionalLayer *buildConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf,
                                                int th_count, std::istream *infile) {
        if (infile != NULL) return new ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, th_count, infile);
        std::vector<float> weights = getPretrained(name + ".weight"), biases = getPretrained(name + ".bias");
        return new ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, th_count, weights, biases);
    }
    // the same with zero padding (xp, yp) (ConvolutionalLayer's padded constructors)
    ConvolutionalLayer *buildConvolutionalLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int xp, int yp,
                                                int th_count, std::istream *infile) {
        if (infile != NULL) return new ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, th_count, infile);
        std::vector<float> weights = getPretrained(name + ".weight"), biases = getPretrained(name + ".bias");
        return new ConvolutionalLayer(name, xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, th_count, weights, biases);
    }
    // cnnBuilder.cpp:54-77
    FullyConnectedLayer *buildFullyConnectedLayer(std::string name, int in_dim, int out_dim, int th_count, std::istream *infile) {
        if (infile != NULL) return new FullyConnectedLayer(name, in_dim, out_dim, th_count, infile);
        std::vector<float> weights = getPretrained(name + ".weight"), biases = getPretrained(name + ".bias");
        return new FullyConnectedLayer(name, in_dim, out_dim, th_count, weights, biases);
    }
    PoolingLayer *buildPoolingLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf) {
        return new PoolingLayer(name, xd, yd, zd, xs, ys, xf, yf);
    }
    AvgPoolingLayer *buildAvgPoolingLayer(std::string name, int xd, int yd, int zd, int xs, int ys, int xf, int yf) {
        return new AvgPoolingLayer(name, xd, yd, zd, xs, ys, xf, yf);
    }
    SquareLayer *buildSquareLayer(std::string name, int th_count) { return new SquareLayer(name, th_count); }
    // mean and 1/sqrt(var + 1e-05), computed in float like the reference (cnnBuilder.cpp:89-105)
    BatchNormLayer *buildBatchNormLayer(std::string name, int num_channels, std::istream *infile) {
        if (infile != NULL) return new BatchNormLayer(name, num_channels, infile);
        std::vector<float> mean = getPretrained(name + ".running_mean"), var = getPretrained(name + ".running_var");
        for (int i = 0; i < num_channels; i++) var[i] = 1 / sqrt(var[i] + 0.00001);
        return new BatchNormLayer(name, num_channels, mean, var);
    }

    // cnnBuilder.cpp:108-179 -- the active (Tiny) block
    Network buildNetwork(std::string file_name = "") { return buildNetwork("Tiny", file_name); }

    Network buildNetwork(const std::string &topology, std::string file_name) {
        Network net;
        buildLayers(net, topology, file_name);
        return net;
    }
    // The same blocks appended to a caller-owned network (e.g. a ShardedNetwork, which cannot be returned by value)
    void buildLayers(Network &net, const std::string &topology, std::string file_name) {
        const int th_count = 40, th_count2 = 50, th_tiny = 32, th_tiny2 = 42;  // cnnBuilder.cpp:109 (accepted and ignored by the layers)
        std::ifstream *infile = NULL;
        if (file_name != "") {
            infile = new std::ifstream(file_name, std::ifstream::binary);
            if (!*infile) { delete infile; throw std::invalid_argument("cannot open encoded network " + file_name); }
        }
        auto add = [&](Layer *l) { net.getLayers().push_back(std::shared_ptr<Layer>(l)); };
        try {
            if (topology == "Tiny") {  // cnnBuilder.cpp:157-169
                add(buildConvolutionalLayer("pool1_features.conv1", 28, 28, 1, 1, 1, 5, 5, 32, th_tiny, infile));
                add(buildAvgPoolingLayer("pool1", 24, 24, 32, 2, 2, 2, 2));
                add(buildConvolutionalLayer("pool2_features.conv2", 12, 12, 32, 1, 1, 5, 5, 64, th_tiny * 2, infile));
                add(buildAvgPoolingLayer("pool2", 8, 8, 64, 2, 2, 2, 2));
                add(buildFullyConnectedLayer("classifier.fc3", 4 * 4 * 64, 512, th_tiny2, infile));
                add(buildFullyConnectedLayer("classifier.fc4", 512, 10, th_tiny2, infile));
            } else if (topology == "Approx" || topology == "WoPad" || topology == "PlainModel" || topology == "PlainModelPadded") {
                // cnnBuilder.cpp:115-134 (avg-pool) / 136-155 (sum-pool); PlainModel: 32x32 zero-bordered input, PlainModelPadded: 28x28 input
                // and conv1 with padding 2 (as PlainModel.h5 was trained); both 14 -> 13 -> 6 -> 5, fc3 1250 -> 500
                const bool avg = topology != "WoPad";
                const int in = topology == "PlainModel" ? 32 : 28, pad = topology == "PlainModelPadded" ? 2 : 0;
                const int c1 = (in + 2 * pad - 5) / 2 + 1, p1 = c1 - 1, c2 = (p1 - 3) / 2 + 1, p2 = c2 - 1;
                add(buildConvolutionalLayer("pool1_features.conv1", in, in, 1, 2, 2, 5, 5, 20, pad, pad, th_count, infile));
                if (avg) add(buildAvgPoolingLayer("pool1", c1, c1, 20, 1, 1, 2, 2)); else add(buildPoolingLayer("pool1", c1, c1, 20, 1, 1, 2, 2));
                add(buildBatchNormLayer("pool1_features.norm1", 20, infile));
                add(buildConvolutionalLayer("pool2_features.conv2", p1, p1, 20, 2, 2, 3, 3, 50, th_count2, infile));
                add(buildSquareLayer("act1", th_count2));
                if (avg) add(buildAvgPoolingLayer("pool2", c2, c2, 50, 1, 1, 2, 2)); else add(buildPoolingLayer("pool2", c2, c2, 50, 1, 1, 2, 2));
                add(buildBatchNormLayer("pool2_features.norm2", 50, infile));
                add(buildFullyConnectedLayer("classifier.fc3", p2 * p2 * 50, 500, th_count, infile));
                add(buildFullyConnectedLayer("classifier.fc4", 500, 10, th_count2, infile));
            } else {
                throw std::invalid_argument("unknown topology " + topology);
            }
        } catch (...) {
            if (infile != NULL) { infile->close(); delete infile; }
            throw;
        }
        if (infile != NULL) { infile->close(); delete infile; }
    }
    // input shape (z, x, y) and number of score ciphertexts of a topology
    static void topologyShape(const std::string &topology, int *zd, int *xd, int *yd, int *outputs) {
        *zd = 1; *xd = *yd = topology == "PlainModel" ? 32 : 28; *outputs = 10;
    }

    // cnnBuilder.cpp:181-196.  Precondition as in the reference: Runtime::init() (their setParameters) has been called.
    Network buildAndSaveNetwork(std::string file_name) { return buildAndSaveNetwork("Tiny", file_name); }
    Network buildAndSaveNetwork(const std::string &topology, std::string file_name) {
        std::ofstream outfile(file_name, std::ofstream::binary);
        if (!outfile) throw std::invalid_argument("cannot write " + file_name);
        Network net = buildNetwork(topology, "");
        for (int i = 0; i < net.getNumLayers(); i++) net.getLayer(i)->savePlaintextParameters(&outfile);
        outfile.close();
        return net;
    }
};

}  // namespace crcnn_b200
