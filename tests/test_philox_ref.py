"""The host transcription of the Philox-mode draws (tests/philox_ref.py) against the device source and the laws.

The GPU tests (test_gpu_philox_draws.py) pin every Philox-mode draw of the kernels to this transcription; these
tests pin the transcription to common.cuh (compiled with nvcc as host code) and to the distributions it samples."""
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import philox_ref as R
from bmm_mcmc_b200 import build as libbuild

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bmm_mcmc_b200", "csrc")

# Random123 known-answer vectors of philox4x32_10: (counter, key, result)
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]

# Host program over common.cuh: "philox" reads n records of 6 uint32 (counter, key) from stdin and writes the four
# words, u53(x, y), u53(z, w), u32_unit(x), u32_unit_f(x) and unit_f(u53(x, y)) of each; "range" walks all 2^24 inputs
# of u32_unit_f and the top inputs of u53 and of its float cast and prints how many values fall outside (0, 1).
HOST_SRC = r"""
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "common.cuh"
using namespace bmm;
int main(int argc, char **argv) {
    if (argc > 1 && !strcmp(argv[1], "range")) {
        long bad_f = 0, bad_53 = 0, bad_53f = 0;
        for (uint32_t h = 0; h < (1u << 24); ++h)
            for (uint32_t lo : {0u, 0xFFu}) { float u = u32_unit_f((h << 8) | lo); bad_f += !(u > 0.f && u < 1.f); }
        for (uint32_t a : {0u, 1u, 0xFFFFFF7Fu, 0xFFFFFF80u, 0xFFFFFFFEu, 0xFFFFFFFFu})
            for (uint32_t b : {0u, 0x7FFu, 0x800u, 0xFFFFF7FFu, 0xFFFFF800u, 0xFFFFFFFFu}) {
                double u = u53(a, b);
                bad_53 += !(u > 0.0 && u < 1.0);
                float f = unit_f(u);
                bad_53f += !(f > 0.f && f < 1.f);
            }
        for (uint32_t a = 0xFFFFFF00u; a != 0u; ++a) { float f = unit_f(u53(a, 0xFFFFFFFFu)); bad_53f += !(f > 0.f && f < 1.f); }
        printf("%ld %ld %ld\n", bad_f, bad_53, bad_53f);
        return 0;
    }
    std::vector<uint32_t> in;
    uint32_t v[6];
    while (fread(v, 4, 6, stdin) == 6) in.insert(in.end(), v, v + 6);
    const size_t n = in.size() / 6;
    std::vector<uint32_t> words(4 * n);
    std::vector<double> dbl(3 * n);
    std::vector<float> flt(2 * n);
    for (size_t i = 0; i < n; ++i) {
        const uint32_t *r = &in[6 * i];
        uint4 o = philox4x32_10(make_uint4(r[0], r[1], r[2], r[3]), make_uint2(r[4], r[5]));
        words[4 * i] = o.x; words[4 * i + 1] = o.y; words[4 * i + 2] = o.z; words[4 * i + 3] = o.w;
        dbl[3 * i] = u53(o.x, o.y); dbl[3 * i + 1] = u53(o.z, o.w); dbl[3 * i + 2] = u32_unit(o.x);
        flt[2 * i] = u32_unit_f(o.x); flt[2 * i + 1] = unit_f(u53(o.x, o.y));
    }
    fwrite(words.data(), 4, words.size(), stdout);
    fwrite(dbl.data(), 8, dbl.size(), stdout);
    fwrite(flt.data(), 4, flt.size(), stdout);
    return 0;
}
"""


@pytest.fixture(scope="module")
def host_prog(tmp_path_factory):
    d = tmp_path_factory.mktemp("philox_host")
    src, exe = d / "host.cu", d / "host"
    src.write_text(HOST_SRC)
    r = subprocess.run([libbuild._nvcc(), "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-I", CSRC, str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


def _run_host(exe, ctr, key):
    rec = np.concatenate([ctr, key], 1).astype("<u4")
    out = subprocess.run([exe], input=rec.tobytes(), capture_output=True, check=True).stdout
    n = len(rec)
    words = np.frombuffer(out, "<u4", 4 * n).reshape(n, 4)
    dbl = np.frombuffer(out, "<f8", 3 * n, offset=16 * n).reshape(n, 3)
    flt = np.frombuffer(out, "<f4", 2 * n, offset=40 * n).reshape(n, 2)
    return words, dbl, flt


def test_known_answers():
    for ctr, key, want in KAT:
        assert tuple(int(v) for v in R.philox(*ctr, *key)) == want


def test_transcription_equals_device_source(host_prog):
    """Philox words and every uniform mapping bit for bit against common.cuh, on 1e5 random counters and keys and on
    the extreme words (the three known-answer inputs included)."""
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2 ** 32, (100_000, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, (100_000, 2), dtype=np.uint64)
    ext = np.array([0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFF00, 0xFFFFFF7F, 0xFFFFFF80, 0xFFFFFFFE, 0xFFFFFFFF], dtype=np.uint64)
    g = np.stack(np.meshgrid(ext, ext, indexing="ij"), -1).reshape(-1, 2)
    ctr = np.concatenate([ctr, np.concatenate([g, g[::-1]], 1), [list(c) for c, _, _ in KAT]])
    key = np.concatenate([key, g, [list(k) for _, k, _ in KAT]])
    words, dbl, flt = _run_host(host_prog, ctr, key)
    ref = R.philox(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], key[:, 0], key[:, 1])
    assert np.array_equal(words, ref)
    assert np.array_equal(words[-3:], np.array([w for _, _, w in KAT], dtype=np.uint32))
    assert np.array_equal(dbl[:, 0], R.u53(ref[:, 0], ref[:, 1]))
    assert np.array_equal(dbl[:, 1], R.u53(ref[:, 2], ref[:, 3]))
    assert np.array_equal(dbl[:, 2], R.u32_unit(ref[:, 0]))
    assert np.array_equal(flt[:, 0], R.u32_unit_f(ref[:, 0]))
    assert np.array_equal(flt[:, 1], np.minimum(R.u53(ref[:, 0], ref[:, 1]).astype(np.float32), R.UF_MAX))


def test_uniforms_strictly_inside_unit_interval(host_prog):
    """u32_unit_f over all 2^24 values of w >> 8, u53 at its extreme inputs and its float cast at every top word:
    no value may reach 0 or 1 (an inverse-CDF draw at u = 1 runs past every category with mass)."""
    out = subprocess.run([host_prog, "range"], capture_output=True, text=True, check=True).stdout.split()
    bad_f, bad_53, bad_53f = (int(v) for v in out)
    assert (bad_f, bad_53, bad_53f) == (0, 0, 0), "common.cuh: %d u32_unit_f, %d u53, %d float-cast values outside (0, 1)" % (
        bad_f, bad_53, bad_53f)
    h = np.arange(1 << 24, dtype=np.uint32) << np.uint32(8)
    for lo in (0, 0xFF):
        u = R.u32_unit_f(h | np.uint32(lo))
        assert u.dtype == np.float32 and u.min() > 0 and u.max() < 1
    assert R.u53(0xFFFFFFFF, 0xFFFFFFFF) < 1.0 and R.u53(0, 0) > 0.0
    assert np.minimum(R.u53(0xFFFFFF80, 0).astype(np.float32), R.UF_MAX) < 1


def test_stream_layout():
    """Counter (attempt, index, stream ^ seed_hi << 8, sweep) and key (seed_lo, chain); two uniforms per block."""
    seed = (7 << 32) | 12345
    st = R.Stream(seed, 9, 4, R.ST_THETA, 21)
    us = [st.uniform() for _ in range(4)]
    b0 = R.philox(0, 21, R.ST_THETA ^ (7 << 8), 4, 12345, 9)
    b1 = R.philox(1, 21, R.ST_THETA ^ (7 << 8), 4, 12345, 9)
    assert us == [R.u53(b0[0], b0[1]), R.u53(b0[2], b0[3]), R.u53(b1[0], b1[1]), R.u53(b1[2], b1[3])]
    w = R.z_words_rows(seed, 3, 2, np.arange(9))
    blk = R.philox(np.arange(3), 0, R.ST_Z ^ (7 << 8), 2, 12345, 3).reshape(-1)
    assert np.array_equal(w, blk[:9])


def _draws(fn, n, stream=R.ST_MISC):
    return np.array([fn(R.Stream(2024, 5, 1, stream, i)) for i in range(n)])


@pytest.mark.parametrize("shape", [0.01, 0.3, 1.0, 2.5, 50.0, 1e4, 1e7])
def test_gamma_law(shape):
    x = _draws(lambda s: s.gamma(shape), 3000)
    p = stats.kstest(x, stats.gamma(shape).cdf).pvalue
    assert p > 1e-3, "Stream.gamma(%g): KS p = %.2e" % (shape, p)


@pytest.mark.parametrize("a,b", [(0.5, 0.5), (1.0, 300.0), (3.5, 0.2), (40.0, 60.0)])
def test_beta_law(a, b):
    x = _draws(lambda s: s.beta(a, b), 3000)
    p = stats.kstest(x, stats.beta(a, b).cdf).pvalue
    assert p > 1e-3, "Stream.beta(%g, %g): KS p = %.2e" % (a, b, p)


@pytest.mark.parametrize("alpha_old,N,K", [(1.0, 1000, 3), (0.2, 100, 2), (5.0, 20077, 32)])
def test_alpha_updates_law(alpha_old, N, K):
    """Both alpha updates against the Escobar-West formula (utils.cpp:6-14) sampled with numpy: two-sample KS."""
    a, b, n = 1.0, 1.0, 2000
    sub = np.array([R.alpha_update_substreams(77, 3, j, alpha_old, a, b, N, K)[0] for j in range(n)])
    seq = np.array([R.update_alpha_seq(R.Stream(77, 3, j, R.ST_ALPHA, 0), alpha_old, a, b, N, K) for j in range(n)])
    rng = np.random.default_rng(3)
    b_eps = b - np.log(rng.beta(alpha_old + 1.0, N, 20000))
    pi1, pi2 = a + K - 1, N * b_eps
    w = pi1 / (pi1 + pi2)
    ref = w * rng.gamma(a + K, 1.0 / b_eps) + (1 - w) * rng.gamma(a + K - 1, 1.0 / b_eps)
    for name, x in (("substreams", sub), ("sequential", seq)):
        p = stats.ks_2samp(x, ref).pvalue
        assert p > 1e-3, "%s alpha update: KS p = %.2e" % (name, p)


def test_icdf_check_flags_wrong_and_zero_weight_draws():
    prob = np.array([[0.5, 0.5, 0.0], [0.2, 0.3, 0.5], [0.2, 0.3, 0.5]])
    u = np.array([0.9999, 0.1, 0.5 + 1e-14])
    bad, exempt, tiny = R.icdf_check(prob, u, np.array([2, 0, 1]), 1e-12)
    assert list(tiny) == [0] and list(bad) == [0] and list(exempt) == [2]
    bad, _, _ = R.icdf_check(prob, u, np.array([1, 1, 2]), 1e-12)
    assert list(bad) == [1]


def test_dp_state_bookkeeping():
    """Used-list order, order-preserving erase and the smallest free label of the DP transcription."""
    X = np.array([[1, 0], [0, 1], [1, 1]])
    st = R.DPState(X, 5)
    prob, pos = st.sweep(1, np.array([0, 0, 1]), 1.0, 0.5, 0.5)
    assert pos.tolist() == [0, 0, 1] and st.used == [0, 1] and st.Nk[:2].tolist() == [2, 1]
    assert prob[0, 0] == 1.0 and np.allclose(prob.sum(1), 1.0) and (prob[1, 2:] == 0).all()
    # sweep 2: row 1 leaves label 0 empty -> erased, label 0 is free again and is the new cluster of row 1's update
    prob, pos = st.sweep(2, np.array([1, 0, 2]), 1.0, 0.5, 0.5)
    assert pos.tolist() == [1, 1, 2]
    assert st.used == [1, 0, 2] and st.Nk[:3].tolist() == [1, 1, 1]
    assert st.S[0].tolist() == [0, 1] and st.S[2].tolist() == [1, 1]
