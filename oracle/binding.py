"""ctypes binding for oracle/libdpfhe_oracle.so (TEST INFRASTRUCTURE ONLY)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libdpfhe_oracle.so")
_lib = None

u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")


def build(force=False):
    src = [os.path.join(_HERE, f) for f in ("dpfhe_oracle.c", "dpfhe_oracle.h", "Makefile")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libdpfhe_oracle.so"], stdout=subprocess.DEVNULL)
    return _SO


def build_ref():
    """oracle/_ref/: the upstream project's examples compiled, unchanged, against include/shim/deeppowers.hpp and libdpfhe.so
    (Makefile target `ref`) when a checkout of deeppowers/deeppowers is at hand: $DEEPPOWERS_SRC, else the checkout
    BASELINE.json names (reference_path).  Returns the directory, or None without a checkout."""
    src = os.environ.get("DEEPPOWERS_SRC")
    if not src:
        with open(os.path.join(_HERE, "..", "BASELINE.json")) as f:
            src = json.load(f).get("reference_path", "")
    src = os.path.abspath(src)
    if not os.path.isdir(os.path.join(src, "examples")):
        return None
    subprocess.check_call(["make", "-C", _HERE, "ref", "DEEPPOWERS_SRC=" + src], stdout=subprocess.DEVNULL)
    return os.path.join(_HERE, "_ref")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        build()
    L = C.CDLL(_SO)
    vp, u64, sz, u32, i32 = C.c_void_p, C.c_uint64, C.c_size_t, C.c_uint, C.c_int
    sig = {
        "dpo_create": (vp, [u32, u32, C.POINTER(u64)]),
        "dpo_destroy": (None, [vp]),
        "dpo_modulus": (u64, [vp, u32]),
        "dpo_psi": (u64, [vp, u32]),
        "dpo_inv_n": (u64, [vp, u32]),
        "dpo_root_powers": (C.POINTER(u64), [vp, u32]),
        "dpo_inv_root_powers": (C.POINTER(u64), [vp, u32]),
        "dpo_mulmod_ref": (u64, [u64, u64, u64]),
        "dpo_mulmod_barrett": (u64, [u64, u64, u64]),
        "dpo_shoup_precompute": (u64, [u64, u64]),
        "dpo_mulmod_shoup": (u64, [u64, u64, u64, u64]),
        "dpo_powmod": (u64, [u64, u64, u64]),
        "dpo_invmod": (u64, [u64, u64]),
        "dpo_is_prime": (i32, [u64]),
        "dpo_ntt_fwd": (None, [vp, u64p, sz]),
        "dpo_ntt_inv": (None, [vp, u64p, sz]),
        "dpo_ntt_fwd_limb_slow": (None, [vp, u32, u64p]),
        "dpo_negacyclic_schoolbook": (None, [vp, u32, u64p, u64p, u64p]),
        "dpo_poly_mul_pointwise": (None, [vp, u64p, u64p, u64p, sz]),
        "dpo_poly_add": (None, [vp, u64p, u64p, u64p, sz]),
        "dpo_ct_tensor": (None, [vp, u64p, u64p, u64p, sz]),
        "dpo_keyswitch": (None, [vp, u64p, u64p, u64p, u64p]),
        "dpo_ct_mul_relin": (None, [vp, u64p, u64p, u64p, u64p, sz]),
        "dpo_ct_mul_plain": (None, [vp, u64p, u64p, u64p, sz]),
        "dpo_ct_mul_plain_inner": (None, [vp, u64p, sz, u64p, sz, u64p, sz]),
        "dpo_rotate": (None, [vp, u64p, u64, u64p, u64p, sz]),
        "dpo_mod_switch_down": (None, [vp, u64p, u64, u64p, sz]),
        "dpo_keyswitch_hybrid": (None, [vp, u64p, u64p, u64, u64p, u64p]),
        "dpo_ct_mul_relin_hybrid": (None, [vp, u64p, u64p, u64p, u64, u64p, sz]),
        "dpo_rotate_hybrid": (None, [vp, u64p, u64, u64p, u64, u64p, sz]),
        "dpo_grouped_digits": (C.c_uint, [vp, C.c_uint]),
        "dpo_mod_down_special": (None, [vp, C.c_uint, u64p, u64, u64p, sz]),
        "dpo_keyswitch_grouped": (None, [vp, C.c_uint, u64p, u64p, u64, u64p, u64p]),
        "dpo_ct_mul_relin_grouped": (None, [vp, C.c_uint, u64p, u64p, u64p, u64, u64p, sz]),
        "dpo_rotate_grouped": (None, [vp, C.c_uint, u64p, u64, u64p, u64, u64p, sz]),
        "dpo_rotate_hoisted_grouped": (None, [vp, C.c_uint, u64p, sz, u64p, u64p, u64, u64p, sz]),
        "dpo_keygen_relin_grouped": (None, [vp, C.c_uint, u64, u64, u64p, u64p]),
        "dpo_keygen_galois_grouped": (None, [vp, C.c_uint, u64, u64, u64p, u64, u64p]),
        "dpo_keygen_relin_hybrid": (None, [vp, u64, u64, u64p, u64p]),
        "dpo_keygen_galois_hybrid": (None, [vp, u64, u64, u64p, u64, u64p]),
        "dpo_galois_perm": (None, [vp, u64, u32p]),
        "dpo_galois_coeff": (None, [vp, u32, u64, u64p, u64p]),
        "dpo_splitmix64": (u64, [u64]),
        "dpo_fill_uniform": (None, [vp, u64, u64, u64p, sz]),
        "dpo_keygen_secret": (None, [vp, u64, u64p]),
        "dpo_keygen_switch": (None, [vp, u64, u64, u64p, u64p, u64p]),
        "dpo_keygen_relin": (None, [vp, u64, u64, u64p, u64p]),
        "dpo_keygen_galois": (None, [vp, u64, u64, u64p, u64, u64p]),
        "dpo_encrypt": (None, [vp, u64, u64, u64p, u64p, u64p]),
        "dpo_phase": (None, [vp, u64p, u64p, u32, u64p]),
        "dpo_max_threads": (i32, []),
        "dpo_num_procs": (i32, []),
        "dpo_time_ct_mul_relin": (C.c_double, [vp, u64p, u64p, u64p, u64p, sz, i32]),
        "dpo_time_ntt_fwd": (C.c_double, [vp, u64p, sz, i32]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _lib = L
    return L


class Oracle:
    """One parameter set (N = 2**logn, L limbs).  Arrays are numpy uint64, layouts as in dpfhe_oracle.h."""

    def __init__(self, logn, L, moduli=None):
        self._l = lib()
        arr = None
        if moduli is not None:
            arr = (C.c_uint64 * L)(*[int(m) for m in moduli])
        self._c = self._l.dpo_create(logn, L, arr)
        if not self._c:
            raise ValueError("dpo_create rejected the parameters")
        self.logn, self.L, self.N = logn, L, 1 << logn
        self.P = self.L * self.N
        self.moduli = [int(self._l.dpo_modulus(self._c, l)) for l in range(L)]
        self.psi = [int(self._l.dpo_psi(self._c, l)) for l in range(L)]

    def __del__(self):
        if getattr(self, "_c", None):
            self._l.dpo_destroy(self._c)
            self._c = None

    # tables
    def root_powers(self, l):
        return np.ctypeslib.as_array(self._l.dpo_root_powers(self._c, l), (self.N,)).copy()

    def inv_root_powers(self, l):
        return np.ctypeslib.as_array(self._l.dpo_inv_root_powers(self._c, l), (self.N,)).copy()

    def inv_n(self, l):
        return int(self._l.dpo_inv_n(self._c, l))

    # transforms (return new arrays)
    def ntt_fwd(self, data):
        d = np.ascontiguousarray(data, dtype=np.uint64).copy()
        self._l.dpo_ntt_fwd(self._c, d.reshape(-1), d.size // self.P)
        return d

    def ntt_inv(self, data):
        d = np.ascontiguousarray(data, dtype=np.uint64).copy()
        self._l.dpo_ntt_inv(self._c, d.reshape(-1), d.size // self.P)
        return d

    def ntt_fwd_limb_slow(self, l, a):
        d = np.ascontiguousarray(a, dtype=np.uint64).copy()
        self._l.dpo_ntt_fwd_limb_slow(self._c, l, d)
        return d

    def schoolbook(self, l, a, b):
        out = np.empty(self.N, dtype=np.uint64)
        self._l.dpo_negacyclic_schoolbook(self._c, l, np.ascontiguousarray(a), np.ascontiguousarray(b), out)
        return out

    def poly_mul_pointwise(self, a, b):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        out = np.empty_like(a)
        self._l.dpo_poly_mul_pointwise(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), out.reshape(-1), a.size // self.P)
        return out

    def poly_add(self, a, b):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        out = np.empty_like(a)
        self._l.dpo_poly_add(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), out.reshape(-1), a.size // self.P)
        return out

    def ct_tensor(self, a, b):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        batch = a.size // (2 * self.P)
        out = np.empty((batch, 3, self.L, self.N), dtype=np.uint64)
        self._l.dpo_ct_tensor(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), out.reshape(-1), batch)
        return out

    def keyswitch(self, d, key):
        c0 = np.empty((self.L, self.N), dtype=np.uint64)
        c1 = np.empty((self.L, self.N), dtype=np.uint64)
        self._l.dpo_keyswitch(self._c, np.ascontiguousarray(d).reshape(-1), np.ascontiguousarray(key).reshape(-1), c0.reshape(-1), c1.reshape(-1))
        return c0, c1

    def ct_mul_relin(self, a, b, evk):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        out = np.empty_like(a)
        self._l.dpo_ct_mul_relin(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), np.ascontiguousarray(evk).reshape(-1), out.reshape(-1), a.size // (2 * self.P))
        return out

    def ct_mul_plain(self, ct, pt):
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        out = np.empty_like(ct)
        self._l.dpo_ct_mul_plain(self._c, ct.reshape(-1), np.ascontiguousarray(pt).reshape(-1), out.reshape(-1), ct.size // (2 * self.P))
        return out

    def ct_mul_plain_inner(self, steps, pts):
        """steps [nb][batch][2][L][N], pts [ng][nb][L][N] -> [ng][batch][2][L][N]"""
        steps = np.ascontiguousarray(steps, dtype=np.uint64)
        pts = np.ascontiguousarray(pts, dtype=np.uint64)
        nb, batch, ng = steps.shape[0], steps.shape[1], pts.shape[0]
        assert pts.shape[1] == nb
        out = np.empty((ng, batch, 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_ct_mul_plain_inner(self._c, steps.reshape(-1), nb, pts.reshape(-1), ng, out.reshape(-1), batch)
        return out

    def rotate(self, ct, galois_elt, gk):
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        out = np.empty_like(ct)
        self._l.dpo_rotate(self._c, ct.reshape(-1), int(galois_elt), np.ascontiguousarray(gk).reshape(-1), out.reshape(-1), ct.size // (2 * self.P))
        return out

    def mod_switch_down(self, polys, t_plain=0):
        """[n][L][N] -> [n][L-1][N]; decrypt the result with Oracle(logn, L-1, moduli[:-1])"""
        x = np.ascontiguousarray(polys, dtype=np.uint64).reshape(-1, self.L, self.N)
        out = np.empty((x.shape[0], self.L - 1, self.N), dtype=np.uint64)
        self._l.dpo_mod_switch_down(self._c, x.reshape(-1), int(t_plain), out.reshape(-1), x.shape[0])
        return out

    # hybrid (special-prime) key switching: this context's last limb is the special prime, data has L-1 limbs
    def keyswitch_hybrid(self, d, key, t_plain=0):
        c0 = np.empty((self.L - 1, self.N), dtype=np.uint64)
        c1 = np.empty((self.L - 1, self.N), dtype=np.uint64)
        self._l.dpo_keyswitch_hybrid(self._c, np.ascontiguousarray(d).reshape(-1), np.ascontiguousarray(key).reshape(-1), int(t_plain),
                                     c0.reshape(-1), c1.reshape(-1))
        return c0, c1

    def ct_mul_relin_hybrid(self, a, b, evk, t_plain=0):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        out = np.empty_like(a)
        self._l.dpo_ct_mul_relin_hybrid(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), np.ascontiguousarray(evk).reshape(-1),
                                        int(t_plain), out.reshape(-1), a.size // (2 * (self.L - 1) * self.N))
        return out

    def rotate_hybrid(self, ct, galois_elt, gk, t_plain=0):
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        out = np.empty_like(ct)
        self._l.dpo_rotate_hybrid(self._c, ct.reshape(-1), int(galois_elt), np.ascontiguousarray(gk).reshape(-1), int(t_plain),
                                  out.reshape(-1), ct.size // (2 * (self.L - 1) * self.N))
        return out

    def keygen_relin_hybrid(self, seed, t, s):
        k = np.empty((self.L - 1, 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_relin_hybrid(self._c, int(seed), int(t), s.reshape(-1), k.reshape(-1))
        return k

    def keygen_galois_hybrid(self, seed, t, s, g):
        k = np.empty((self.L - 1, 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_galois_hybrid(self._c, int(seed), int(t), s.reshape(-1), int(g), k.reshape(-1))
        return k

    # grouped hybrid key switching: the last K limbs are special primes, data has L-K limbs, keys have ceil((L-K)/K) digits
    def grouped_digits(self, K):
        return int(self._l.dpo_grouped_digits(self._c, int(K)))

    def mod_down_special(self, K, polys, t_plain=0):
        x = np.ascontiguousarray(polys, dtype=np.uint64).reshape(-1, self.L, self.N)
        out = np.empty((x.shape[0], self.L - K, self.N), dtype=np.uint64)
        self._l.dpo_mod_down_special(self._c, int(K), x.reshape(-1), int(t_plain), out.reshape(-1), x.shape[0])
        return out

    def keyswitch_grouped(self, K, d, key, t_plain=0):
        c0 = np.empty((self.L - K, self.N), dtype=np.uint64)
        c1 = np.empty((self.L - K, self.N), dtype=np.uint64)
        self._l.dpo_keyswitch_grouped(self._c, int(K), np.ascontiguousarray(d).reshape(-1), np.ascontiguousarray(key).reshape(-1), int(t_plain),
                                      c0.reshape(-1), c1.reshape(-1))
        return c0, c1

    def ct_mul_relin_grouped(self, K, a, b, evk, t_plain=0):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        out = np.empty_like(a)
        self._l.dpo_ct_mul_relin_grouped(self._c, int(K), a.reshape(-1), np.ascontiguousarray(b).reshape(-1),
                                         np.ascontiguousarray(evk).reshape(-1), int(t_plain), out.reshape(-1),
                                         a.size // (2 * (self.L - K) * self.N))
        return out

    def rotate_grouped(self, K, ct, galois_elt, gk, t_plain=0):
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        out = np.empty_like(ct)
        self._l.dpo_rotate_grouped(self._c, int(K), ct.reshape(-1), int(galois_elt), np.ascontiguousarray(gk).reshape(-1), int(t_plain),
                                   out.reshape(-1), ct.size // (2 * (self.L - K) * self.N))
        return out

    def rotate_hoisted_grouped(self, K, ct, galois, gks, t_plain=0):
        """ct [batch][2][L-K][N], gks [n_rot][dnum][2][L][N] -> [n_rot][batch][2][L-K][N]"""
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        g = np.ascontiguousarray(galois, dtype=np.uint64)
        batch = ct.size // (2 * (self.L - K) * self.N)
        out = np.empty((len(g), batch) + ct.shape[-3:], dtype=np.uint64)
        self._l.dpo_rotate_hoisted_grouped(self._c, int(K), ct.reshape(-1), len(g), g, np.ascontiguousarray(gks, dtype=np.uint64).reshape(-1),
                                           int(t_plain), out.reshape(-1), batch)
        return out

    def keygen_relin_grouped(self, K, seed, t, s):
        k = np.empty((self.grouped_digits(K), 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_relin_grouped(self._c, int(K), int(seed), int(t), s.reshape(-1), k.reshape(-1))
        return k

    def keygen_galois_grouped(self, K, seed, t, s, g):
        k = np.empty((self.grouped_digits(K), 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_galois_grouped(self._c, int(K), int(seed), int(t), s.reshape(-1), int(g), k.reshape(-1))
        return k

    def galois_perm(self, g):
        p = np.empty(self.N, dtype=np.uint32)
        self._l.dpo_galois_perm(self._c, int(g), p)
        return p

    def galois_coeff(self, l, g, a):
        out = np.empty(self.N, dtype=np.uint64)
        self._l.dpo_galois_coeff(self._c, l, int(g), np.ascontiguousarray(a, dtype=np.uint64), out)
        return out

    def galois_elt(self, k):
        """Galois element 5^k mod 2N (k may be negative)."""
        two_n = 2 * self.N
        return pow(5, k % (self.N // 2), two_n)

    # synthetic data
    def fill_uniform(self, seed, n_polys, first_poly=0):
        d = np.empty((n_polys, self.L, self.N), dtype=np.uint64)
        self._l.dpo_fill_uniform(self._c, int(seed), int(first_poly), d.reshape(-1), n_polys)
        return d

    # scheme
    def keygen_secret(self, seed):
        s = np.empty((self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_secret(self._c, int(seed), s.reshape(-1))
        return s

    def keygen_relin(self, seed, t, s):
        k = np.empty((self.L, 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_relin(self._c, int(seed), int(t), s.reshape(-1), k.reshape(-1))
        return k

    def keygen_galois(self, seed, t, s, g):
        k = np.empty((self.L, 2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_keygen_galois(self._c, int(seed), int(t), s.reshape(-1), int(g), k.reshape(-1))
        return k

    def encrypt(self, seed, t, s, msg):
        ct = np.empty((2, self.L, self.N), dtype=np.uint64)
        self._l.dpo_encrypt(self._c, int(seed), int(t), s.reshape(-1), np.ascontiguousarray(msg, dtype=np.uint64), ct.reshape(-1))
        return ct

    def phase(self, s, ct):
        ct = np.ascontiguousarray(ct, dtype=np.uint64)
        n_comp = ct.size // self.P
        ph = np.empty((self.L, self.N), dtype=np.uint64)
        self._l.dpo_phase(self._c, s.reshape(-1), ct.reshape(-1), n_comp, ph.reshape(-1))
        return ph

    def decrypt(self, s, ct, t):
        """CRT-lift the phase to (-Q/2, Q/2] and reduce mod t (python big ints)."""
        ph = self.phase(s, ct)
        Q = 1
        for q in self.moduli:
            Q *= q
        coef = []
        for q in self.moduli:
            Qi = Q // q
            coef.append(Qi * pow(Qi, -1, q))
        out = np.empty(self.N, dtype=np.uint64)
        cols = [ph[l].tolist() for l in range(self.L)]
        for n in range(self.N):
            v = 0
            for l in range(self.L):
                v += cols[l][n] * coef[l]
            v %= Q
            if v > Q // 2:
                v -= Q
            out[n] = v % t
        return out

    # timing (bench cpu_baseline)
    def max_threads(self):
        return int(self._l.dpo_max_threads())

    def host_threads(self):
        """all the threads the timing helpers can use: the processors OpenMP sees, even when a launcher (torchrun sets
        OMP_NUM_THREADS=1 per rank) capped the default team size; 1 when the oracle was built without OpenMP"""
        return max(int(self._l.dpo_num_procs()), int(self._l.dpo_max_threads()))

    def time_ct_mul_relin(self, a, b, evk, threads=0, out=None):
        """seconds of one dpo_ct_mul_relin over the batch; pass `out` to reuse a touched output buffer (a fresh one makes the
        timed region pay the page faults of first-touching it)"""
        a = np.ascontiguousarray(a, dtype=np.uint64)
        if out is None:
            out = np.empty_like(a)
        assert out.shape == a.shape and out.dtype == np.uint64 and out.flags.c_contiguous
        return float(self._l.dpo_time_ct_mul_relin(self._c, a.reshape(-1), np.ascontiguousarray(b).reshape(-1), np.ascontiguousarray(evk).reshape(-1), out.reshape(-1), a.size // (2 * self.P), threads)), out

    def time_ntt_fwd(self, data, threads=0):
        d = np.ascontiguousarray(data, dtype=np.uint64).copy()
        return float(self._l.dpo_time_ntt_fwd(self._c, d.reshape(-1), d.size // self.P, threads)), d
