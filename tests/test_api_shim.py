"""Row f-1/f-3: the reference's own examples compile and link, unchanged, against include/shim/deeppowers.hpp +
libdpfhe.so (build() compiles them into oracle/_ref where a checkout of the reference is at hand); the Model API's
encrypted route (DPFHEv1 files in, GPU ct x ct, file out) matches the oracle."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_BIN = os.path.join(ROOT, "oracle", "_ref")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def _link(src, exe):
    import deeppowers_b200
    deeppowers_b200.load_library()
    lib_dir = os.path.join(ROOT, "deeppowers_b200")
    subprocess.check_call([GXX, "-std=c++17", "-I", os.path.join(ROOT, "include", "shim"), "-I", os.path.join(ROOT, "include"), src,
                           "-L", lib_dir, "-ldpfhe", "-Wl,-rpath," + lib_dir, "-pthread", "-o", exe])


@pytest.fixture(scope="module")
def ref_bin(oracle_mod):
    """oracle/_ref, (re)built here when a checkout of the reference is at hand, else as build() left it"""
    import deeppowers_b200
    deeppowers_b200.load_library()
    d = oracle_mod.build_ref() or REF_BIN
    if not os.path.isdir(d):
        pytest.skip("no checkout of the reference, and oracle/_ref was not built from one")
    return d


@pytest.mark.parametrize("name", ["basic_generation", "quantization_example", "batch_generation", "stream_generation"])
def test_reference_examples_link_unchanged(ref_bin, name):
    exe = os.path.join(ref_bin, name)       # compiled where it lies by oracle/Makefile (target ref); nothing is copied
    assert os.access(exe, os.X_OK), exe + " was not built"
    if name in ("basic_generation", "batch_generation"):
        r = subprocess.run([exe], input="Hello there\n", capture_output=True, text=True, timeout=60)
        assert r.returncode == 0, r.stderr
        assert "Hello there" in r.stdout or "Generated" in r.stdout


def test_wire_hybrid_key_roundtrip(tmp_path, oracle_mod):
    from deeppowers_b200 import wire
    o = oracle_mod.Oracle(12, 3)
    key = o.fill_uniform(6, 4).reshape(2, 2, 3, o.N)      # [L-1][2][L][N]
    p = str(tmp_path / "hk.dpfhe")
    wire.write(p, 12, 3, wire.HYBRID_SWITCH_KEY, 1, o.moduli, key)
    hdr, data = wire.read(p)
    assert hdr["kind"] == wire.HYBRID_SWITCH_KEY and hdr["moduli"] == o.moduli and np.array_equal(data.reshape(key.shape), key)


def test_wire_grouped_key_roundtrip(tmp_path, oracle_mod):
    """kind 5: a grouped hybrid key announces its number of special primes in `count`; C++ and Python agree on the payload size"""
    from deeppowers_b200 import wire
    o = oracle_mod.Oracle(12, 5)
    key = o.fill_uniform(6, 4).reshape(2, 2, 5, o.N)      # K = 2: ceil(3 / 2) = 2 digits, [2][2][L][N]
    p = str(tmp_path / "gk.dpfhe")
    wire.write(p, 12, 5, wire.GROUPED_SWITCH_KEY, 2, o.moduli, key)
    hdr, data = wire.read(p)
    assert hdr["kind"] == wire.GROUPED_SWITCH_KEY and hdr["count"] == 2 and np.array_equal(data.reshape(key.shape), key)
    with pytest.raises(ValueError):
        wire.write(p, 12, 5, wire.GROUPED_SWITCH_KEY, 3, o.moduli, key)      # 2K > L
    src = str(tmp_path / "w.cpp")
    with open(src, "w") as f:
        f.write('#include <dpfhe_wire.hpp>\n#include <iostream>\nint main(int, char **v) { std::vector<std::uint64_t> d; '
                'auto h = deeppowers::api::fhe::read_wire_file(v[1], d); std::cout << h.kind << " " << h.count << " " << d.size() << " " << d[5]; }\n')
    exe = str(tmp_path / "w")
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
    out = subprocess.run([exe, p], capture_output=True, text=True, check=True).stdout.split()
    assert out == ["5", "2", str(key.size), str(int(key.reshape(-1)[5]))]


def test_wire_format_roundtrip(tmp_path, oracle_mod):
    from deeppowers_b200 import wire
    o = oracle_mod.Oracle(12, 2)
    ct = o.fill_uniform(5, 6).reshape(3, 2, 2, o.N)
    p = str(tmp_path / "x.dpfhe")
    wire.write(p, 12, 2, wire.CIPHERTEXTS, 3, o.moduli, ct)
    hdr, data = wire.read(p)
    assert hdr == {"log_n": 12, "n_limbs": 2, "kind": 1, "form": 1, "count": 3, "moduli": o.moduli}
    assert np.array_equal(data.reshape(ct.shape), ct)
    assert os.path.getsize(p) == 160 + ct.size * 8
    with open(p, "r+b") as f:
        f.write(b"XXXX")
    with pytest.raises(ValueError):
        wire.read(p)


@pytest.mark.gpu
def test_model_api_encrypted_route_matches_oracle(tmp_path, oracle_mod):
    from deeppowers_b200 import wire
    exe = str(tmp_path / "encrypted_job")
    _link(os.path.join(ROOT, "examples", "encrypted_job.cpp"), exe)
    log_n, L, B = 12, 3, 5
    o = oracle_mod.Oracle(log_n, L)
    s = o.keygen_secret(1)
    evk = o.keygen_relin(2, 65537, s)
    a = o.fill_uniform(3, 2 * B).reshape(B, 2, L, o.N)
    b = o.fill_uniform(4, 2 * B).reshape(B, 2, L, o.N)
    fa, fb, fk, fo = (str(tmp_path / n) for n in ("a.dpfhe", "b.dpfhe", "k.dpfhe", "o.dpfhe"))
    wire.write(fa, log_n, L, wire.CIPHERTEXTS, B, o.moduli, a)
    wire.write(fb, log_n, L, wire.CIPHERTEXTS, B, o.moduli, b)
    wire.write(fk, log_n, L, wire.SWITCH_KEY, 1, o.moduli, evk)
    r = subprocess.run([exe, fa, fb, fk, fo, str(log_n), str(L)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    hdr, data = wire.read(fo)
    assert hdr["count"] == B and hdr["kind"] == wire.CIPHERTEXTS
    assert np.array_equal(data.reshape(a.shape), o.ct_mul_relin(a, b, evk))
    # the same job sharded over every visible GPU (config 5's route through the Model API)
    os.remove(fo)
    r = subprocess.run([exe, fa, fb, fk, fo, str(log_n), str(L), "all"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "GPU" in r.stdout, r.stderr
    hdr, data = wire.read(fo)
    assert np.array_equal(data.reshape(a.shape), o.ct_mul_relin(a, b, evk))


@pytest.mark.gpu
def test_model_api_encrypted_route_with_special_prime_keys(tmp_path, oracle_mod):
    """the same Model API route with a grouped relinearisation key file (wire kind 5, two special primes) and a hybrid one (kind 4)"""
    from deeppowers_b200 import wire
    exe = str(tmp_path / "encrypted_job")
    _link(os.path.join(ROOT, "examples", "encrypted_job.cpp"), exe)
    log_n, B, t = 12, 4, 65537
    for L, K, kind in ((6, 2, wire.GROUPED_SWITCH_KEY), (4, 1, wire.HYBRID_SWITCH_KEY)):
        o = oracle_mod.Oracle(log_n, L)
        Lq = L - K
        oq = oracle_mod.Oracle(log_n, Lq, o.moduli[:Lq])
        s = o.keygen_secret(1)
        evk = o.keygen_relin_grouped(K, 2, t, s)
        a = oq.fill_uniform(3, 2 * B).reshape(B, 2, Lq, o.N)
        b = oq.fill_uniform(4, 2 * B).reshape(B, 2, Lq, o.N)
        fa, fb, fk, fo = (str(tmp_path / (n + str(K))) for n in ("a.dpfhe", "b.dpfhe", "k.dpfhe", "o.dpfhe"))
        wire.write(fa, log_n, Lq, wire.CIPHERTEXTS, B, oq.moduli, a)
        wire.write(fb, log_n, Lq, wire.CIPHERTEXTS, B, oq.moduli, b)
        wire.write(fk, log_n, L, kind, K if kind == wire.GROUPED_SWITCH_KEY else 1, o.moduli, evk)
        r = subprocess.run([exe, fa, fb, fk, fo, str(log_n), str(L), "one", str(t)], capture_output=True, text=True, timeout=120)
        assert r.returncode == 0 and "special prime" in r.stdout, r.stderr
        hdr, data = wire.read(fo)
        assert hdr["count"] == B and hdr["n_limbs"] == Lq
        assert np.array_equal(data.reshape(a.shape), o.ct_mul_relin_grouped(K, a, b, evk, t))


def test_wire_reader_rejects_forged_headers(tmp_path, oracle_mod):
    """A header is untrusted input (ADVICE r01): a count that wraps the size computation, a count larger than the file, an
    unknown kind or trailing bytes must all be refused by the C++ reader the shim uses (include/dpfhe_wire.hpp)."""
    import struct
    from deeppowers_b200 import wire
    o = oracle_mod.Oracle(12, 1)
    ct = o.fill_uniform(5, 2).reshape(1, 2, 1, o.N)
    good = str(tmp_path / "good.dpfhe")
    wire.write(good, 12, 1, wire.CIPHERTEXTS, 1, o.moduli, ct)
    raw = open(good, "rb").read()

    def forged(name, count=None, kind=None, extra=b""):
        hdr = list(wire._HDR.unpack(raw[:160]))
        if count is not None:
            hdr[5] = count
        if kind is not None:
            hdr[3] = kind
        path = str(tmp_path / name)
        with open(path, "wb") as f:
            f.write(wire._HDR.pack(*hdr) + raw[160:] + extra)
        return path

    bad = [forged("wrap.dpfhe", count=(1 << 48) + 1), forged("big.dpfhe", count=2), forged("kind.dpfhe", kind=9),
           forged("tail.dpfhe", extra=b"\0" * 8), forged("huge.dpfhe", count=(1 << 64) - 1)]
    for path in bad:
        with pytest.raises(ValueError):
            wire.read(path)
    src = tmp_path / "rd.cpp"
    src.write_text("""
#include "dpfhe_wire.hpp"
#include <iostream>
int main(int argc, char **argv) {
    using namespace deeppowers::api::fhe;
    int refused = 0;
    for (int i = 1; i < argc; ++i) {
        std::vector<std::uint64_t> payload;
        try { WireHeader h = read_wire_file(argv[i], payload); std::cout << "accepted " << argv[i] << " count " << h.count << " words " << payload.size() << "\\n"; }
        catch (const std::runtime_error &e) { ++refused; }
    }
    std::cout << "refused " << refused << "\\n";
    return 0;
}
""")
    exe = str(tmp_path / "rd")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    out = subprocess.run([exe, good] + bad, capture_output=True, text=True, check=True).stdout
    assert "accepted " + good in out and "refused %d" % len(bad) in out, out
