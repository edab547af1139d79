"""CPU: zero-padded convolutions without a GPU.

(1) The pooled grid with padding (crcnn_conv_pool_bn_forward_padded, DESIGN.md 4.5), stated with the oracle's primitives and exact integer
arithmetic: window sums S over the PADDED extent whose border entries are the zero ciphertext (an entry -1 of the index table adds
nothing; a window of border entries only is the zero ciphertext), then one weighted sum at the combined stride with the folded weights
and the unchanged folded bias |window| * B, equal the oracle's layer-by-layer conv -> pool -> batch-norm on the zero-bordered input.
(2) The C++ layer: CnnBuilder::topologyShape("PlainModelPadded"), the padded output size of ConvolutionalLayer, and refused padding.
(3) The Python topology table of the padded network."""
import os
import subprocess

import numpy as np
import pytest

from util import PRIMES, T_FOR_N, random_cts
from oracle.port import Oracle
from test_fold_identities import N, _mod_rows, _ntt_delta_plain, _ntt_plain, _weighted_sum_ntt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def env():
    primes, t = PRIMES[N], T_FOR_N[N]
    return primes, t, Oracle(N, primes, t), np.random.default_rng(78)


# (xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, pxs, pys, pxf, pyf): PlainModel's conv1 block (5x5 / 2, padding 2, 2x2 / 1 pooling) on a small
# input, and stride 1 with padding 2 (the first window sums of S lie entirely in the border)
GEOMETRIES = [(5, 5, 1, 2, 2, 5, 5, 2, 2, 2, 1, 1, 2, 2), (3, 4, 2, 1, 1, 3, 3, 1, 2, 1, 1, 1, 2, 2)]


@pytest.mark.parametrize("geo", GEOMETRIES)
def test_padded_conv_pool_bn_on_the_pooled_grid(env, geo):
    primes, t, orc, rng = env
    xd, yd, zd, xs, ys, xf, yf, nf, xp, yp, pxs, pys, pxf, pyf = geo
    xe, ye = xd + 2 * xp, yd + 2 * yp
    cxo, cyo = (xe - xf) // xs + 1, (ye - yf) // ys + 1
    pxo, pyo = (cxo - pxf) // pxs + 1, (cyo - pyf) // pys + 1
    Rp, R = pxf * pyf, zd * xf * yf
    f = lambda k: rng.uniform(-1, 1, size=k).astype(np.float32)
    wv, bv, mv, vv = f(nf * R), f(nf), f(nf), rng.uniform(-3, 3, size=nf).astype(np.float32)
    wp, bp, mp, vp = (orc.encode_many(v) for v in (wv, bv, mv, vv))
    d, cc = orc.encode(1.0 / Rp)
    x = random_cts(rng, N, primes, zd * xd * yd)
    ct = x.shape[1:]
    xb = np.pad(x.reshape(zd, xd, yd, *ct), [(0, 0), (xp, xp), (yp, yp)] + [(0, 0)] * len(ct)).reshape(-1, *ct)
    conv = orc.conv(xb, xe, ye, zd, xs, ys, xf, yf, nf, wp, bp).reshape(nf * cxo * cyo, *ct)
    want = orc.bn(orc.pool(conv, cxo, cyo, nf, pxs, pys, pxf, pyf, d, cc), nf, pxo, pyo, mp, vp).reshape(nf, pxo, pyo, *ct)
    # S over the padded extent from the UNBORDERED input: index -1 (border) adds nothing, an all-border window is the zero ciphertext
    xi = x.reshape(zd, xd, yd, *ct)
    sxd, syd = xe - (pxf - 1) * xs, ye - (pyf - 1) * ys
    S = np.zeros((zd, sxd, syd) + ct, dtype=np.uint64)
    empty = 0
    for z in range(zd):
        for u in range(sxd):
            for v in range(syd):
                win = [xi[z, u + a * xs - xp, v + b * ys - yp] for a in range(pxf) for b in range(pyf)
                       if 0 <= u + a * xs - xp < xd and 0 <= v + b * ys - yp < yd]
                if win:
                    S[z, u, v] = orc.add_many(np.stack(win))
                else:
                    empty += 1
    assert empty > 0 or geo == GEOMETRIES[0]
    s_ntt = _ntt_plain(orc, d[:cc] if cc else d)
    for k in range(nf):
        v_ntt = _ntt_plain(orc, vp[k])
        C = _mod_rows(s_ntt * v_ntt, primes)
        D = _mod_rows(_ntt_delta_plain(orc, mp[k], primes) * v_ntt, primes)
        Wf = [_mod_rows(_ntt_plain(orc, wp[k * R + r]) * C, primes) for r in range(R)]
        Bf = _mod_rows(Rp * _ntt_delta_plain(orc, bp[k], primes) * C - D, primes)      # |window| * B: the border carries the bias too
        for i in range(pxo):
            for j in range(pyo):
                cols = [S[z, i * pxs * xs + kx, j * pys * ys + ky] for z in range(zd) for kx in range(xf) for ky in range(yf)]
                got = _weighted_sum_ntt(orc, primes, np.stack(cols), Wf, Bf)
                assert np.array_equal(got, want[k, i, j]), (geo, k, i, j)


PROG = r'''
#include <cstdio>
#include "crcnn_b200/cpp/cnn_builder.hpp"
using namespace crcnn_b200;
int main() {
    int z, x, y, o;
    CnnBuilder::topologyShape("PlainModelPadded", &z, &x, &y, &o);
    std::printf("shape %d %d %d %d\n", z, x, y, o);
    plaintext4D f;
    std::vector<Plaintext> b;
    ConvolutionalLayer c1("conv1", 28, 28, 1, 2, 2, 5, 5, 20, 2, 2, 40, f, b);
    ConvolutionalLayer c2("conv", 5, 6, 3, 1, 2, 3, 3, 4, 2, 1, 1, f, b);
    ConvolutionalLayer c3("conv", 28, 28, 1, 2, 2, 5, 5, 20, 40, f, b);
    std::printf("out %d %d %d %d %d %d %d %d %d\n", c1.xo, c1.yo, c1.zo, c2.xo, c2.yo, c3.xo, c3.yo, c3.xp, c3.yp);
    int refused = 0;
    for (int p : {-1, 5, 6}) {
        try { ConvolutionalLayer bad("bad", 28, 28, 1, 2, 2, 5, 5, 20, p, 0, 40, f, b); } catch (const std::invalid_argument &) { refused++; }
        try { ConvolutionalLayer bad("bad", 28, 28, 1, 2, 2, 5, 5, 20, 0, p, 40, f, b); } catch (const std::invalid_argument &) { refused++; }
    }
    std::printf("refused %d\n", refused);
    return 0;
}
'''


def test_padded_layer_geometry_cpp(tmp_path):
    src, exe = tmp_path / "t.cpp", tmp_path / "t"
    src.write_text(PROG)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + ROOT, "-o", str(exe), str(src), "-L" + os.path.join(ROOT, "crcnn_b200"),
                           "-lcrcnn_b200", "-Wl,-rpath," + os.path.join(ROOT, "crcnn_b200")])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-500:] + out.stderr[-500:]
    lines = out.stdout.strip().splitlines()
    assert "shape 1 28 28 10" in lines
    # (28 + 4 - 5) / 2 + 1 = 14; (5 + 4 - 3) / 1 + 1 = 7, (6 + 2 - 3) / 2 + 1 = 3; the reference's constructor: no padding, 12 x 12
    assert "out 14 14 20 7 3 12 12 0 0" in lines
    assert "refused 6" in lines


def test_padded_topology_table():
    from crcnn_b200 import nets
    assert "PlainModelPadded" not in nets.TOPOLOGIES
    padded, plain = nets.topology("PlainModelPadded"), nets.topology("PlainModel")
    assert padded["input"] == (1, 28, 28) and padded["layers"][1:] == plain["layers"][1:]
    conv1 = padded["layers"][0]
    assert conv1[:2] == plain["layers"][0][:2] and conv1[10:] == (2, 2)
    assert nets.conv_out(conv1) == nets.conv_out(plain["layers"][0]) == (14, 14)
    assert nets.layer_io_counts(conv1) == (784, 20 * 14 * 14) and nets.layer_terms(conv1) == nets.layer_terms(plain["layers"][0])
    assert sorted(nets.load_weights("PlainModelPadded")) == sorted(nets.load_weights("PlainModel"))
