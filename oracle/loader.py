"""ctypes loader for the tier-1 C oracle (oracle/c/ark_oracle.c).  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libark_oracle.so")
_lib = None


def _cpu_tag() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _writable(path: str) -> bool:
    while not os.path.exists(path):
        path = os.path.dirname(path)
    return os.access(path, os.W_OK)


def build(force: bool = False) -> str:
    """(Re)build with -march=native; rebuilt when the source is newer or the host CPU changed
    (a checkout may be built on one machine and run on another).  The library goes to oracle/_build, or, when the
    tree is read-only, to a per-user directory under the system temporary directory keyed by source and host CPU."""
    src = os.path.join(_HERE, "c", "ark_oracle.c")
    so, stamp = _SO, os.path.join(_HERE, "_build", "host.txt")
    tag = _cpu_tag()

    def fresh():
        same_host = os.path.exists(stamp) and open(stamp).read() == tag
        return not force and same_host and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src)

    if fresh():
        return so
    if not _writable(os.path.dirname(so)):
        import hashlib
        import tempfile
        key = hashlib.sha256(open(src, "rb").read() + tag.encode()).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"dplonk-oracle-{os.getuid()}-{key}")
        so, stamp = os.path.join(out_dir, "libark_oracle.so"), os.path.join(out_dir, "host.txt")
        if fresh():
            return so
    import fcntl
    os.makedirs(os.path.dirname(so), exist_ok=True)
    with open(so + ".lock", "w") as lock:           # several processes of one test may get here together
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not fresh():
            subprocess.check_call(["make", "-s", "-B", "-C", _HERE, f"OUT={so}"])
            with open(stamp, "w") as f:
                f.write(tag)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        u64, p, i = C.c_uint64, C.c_void_p, C.c_int
        sig = {
            "orc_fft_in_place": (None, [p, u64, i]),
            "orc_coset_fft_in_place": (None, [p, u64, i]),
            "orc_fft1_helper": (None, [p, u64, i, i, u64, i]),
            "orc_fft2_helper": (None, [p, u64, i, i, u64, i]),
            "orc_distributed_fft": (None, [p, p, u64, i, i, u64, i]),
            "orc_fr_mul": (None, [p, p, p]),
            "orc_fr_add": (None, [p, p, p]),
            "orc_fr_sub": (None, [p, p, p]),
            "orc_fq_mul": (None, [p, p, p]),
            "orc_fq_add": (None, [p, p, p]),
            "orc_fq_sub": (None, [p, p, p]),
            "orc_fr_into_repr": (None, [p, p, u64]),
            "orc_fr_from_repr": (None, [p, p, u64]),
            "orc_g1_normalize": (None, [p, p]),
            "orc_g1_add": (None, [p, p, p]),
            "orc_g1_mul": (None, [p, p, p]),
            "orc_g1_generator": (None, [p]),
            "orc_gen_fr": (None, [u64, u64, p, i]),
            "orc_gen_bases": (None, [u64, u64, u64, i, p]),
            "orc_msm_window_c": (u64, [u64]),
            "orc_msm_work_adds": (C.c_double, [u64, u64]),
            "orc_msm": (None, [p, p, u64, p]),
            "orc_commit": (None, [p, u64, p, u64, p]),
            "orc_num_threads": (i, []),
            "orc_set_num_threads": (None, [i]),
            "orc_ntt_outputs_at": (None, [p, u64, u64, p, u64, i, i, p]),
            "orc_fr_dot_u64": (None, [p, p, u64, p]),
            "orc_ntt_output_at": (None, [p, u64, u64, i, i, p]),
            "orc_perm_product": (i, [p, p, p, u64, u64, p, p, p]),
            "orc_quotient_evals": (None, [p, p, p, p, p, p, p, p, p, u64, u64, p]),
            "orc_fr_vec_op": (None, [p, p, p, u64, i]),
            "orc_gen_srs": (None, [p, u64, p]),
            "orc_g1_compress": (None, [p, p]),
            "orc_g1_decompress": (i, [p, p, i]),
            "orc_g1_point_outside_subgroup": (i, [p]),
            "orc_poly_eval": (None, [p, u64, p, p]),
            "orc_poly_lincomb": (None, [p, p, p, u64, p, u64]),
            "orc_poly_div_linear": (None, [p, u64, p, p]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _ptr(a: np.ndarray):
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


# ---- numpy-level helpers (arrays are uint64 [n,4] for Fr, uint8 [n,104] bases, uint8[144] points)
def gen_fr(seed: int, n: int, montgomery: bool = True) -> np.ndarray:
    out = np.empty((n, 4), dtype=np.uint64)
    lib().orc_gen_fr(seed, n, _ptr(out), int(montgomery))
    return out


def gen_bases(seed: int, n: int, distinct: int = 2048, with_infinity: bool = True) -> np.ndarray:
    out = np.zeros((n, 104), dtype=np.uint8)
    lib().orc_gen_bases(seed, n, distinct, int(with_infinity), _ptr(out))
    return out


def fft(x: np.ndarray, inverse: bool = False, coset: bool = False) -> np.ndarray:
    y = np.ascontiguousarray(x, dtype=np.uint64).copy()
    n = y.shape[0]
    (lib().orc_coset_fft_in_place if coset else lib().orc_fft_in_place)(_ptr(y), n, int(inverse))
    return y


def fft1_helper(v, i, is_coset, is_inv, domain_size, as_written=False):
    y = np.ascontiguousarray(v, dtype=np.uint64).copy()
    lib().orc_fft1_helper(_ptr(y), i, int(is_coset), int(is_inv), domain_size, int(as_written))
    return y


def fft2_helper(v, i, is_coset, is_inv, domain_size, as_written=False):
    y = np.ascontiguousarray(v, dtype=np.uint64).copy()
    lib().orc_fft2_helper(_ptr(y), i, int(is_coset), int(is_inv), domain_size, int(as_written))
    return y


def distributed_fft(x, domain_size, is_inv, is_coset, n_workers=1, as_written=False):
    xin = np.zeros((domain_size, 4), dtype=np.uint64)
    xin[: x.shape[0]] = x
    out = np.empty_like(xin)
    lib().orc_distributed_fft(_ptr(xin), _ptr(out), domain_size, int(is_inv), int(is_coset), n_workers, int(as_written))
    return out


def ntt_output_at(x: np.ndarray, k: int, inverse: bool, coset: bool) -> np.ndarray:
    """element k of the (coset) (i)NTT of x, in O(n) (Horner)"""
    x = np.ascontiguousarray(x, dtype=np.uint64)
    out = np.zeros(4, dtype=np.uint64)
    lib().orc_ntt_output_at(_ptr(x), x.shape[0], k, int(inverse), int(coset), _ptr(out))
    return out


def ntt_outputs_at(x: np.ndarray, domain_size: int, ks, inverse: bool, coset: bool) -> np.ndarray:
    """elements ks of the domain_size-point (coset) (i)NTT of x zero-padded to the domain, O(len(x)) each"""
    x = np.ascontiguousarray(x, dtype=np.uint64)
    kk = np.ascontiguousarray(ks, dtype=np.uint64)
    out = np.zeros((kk.shape[0], 4), dtype=np.uint64)
    lib().orc_ntt_outputs_at(_ptr(x), x.shape[0], domain_size, _ptr(kk), kk.shape[0], int(inverse), int(coset), _ptr(out))
    return out


def fr_dot_u64(scalars_canonical: np.ndarray, ks: np.ndarray) -> np.ndarray:
    """sum_i s_i * k_i mod r (canonical), s canonical Fr, k 64-bit"""
    s = np.ascontiguousarray(scalars_canonical, dtype=np.uint64)
    kk = np.ascontiguousarray(ks, dtype=np.uint64)
    out = np.zeros(4, dtype=np.uint64)
    lib().orc_fr_dot_u64(_ptr(s), _ptr(kk), kk.shape[0], _ptr(out))
    return out


def g1_generator() -> np.ndarray:
    out = np.zeros(104, dtype=np.uint8)
    lib().orc_g1_generator(_ptr(out))
    return out


def set_num_threads(n: int) -> None:
    lib().orc_set_num_threads(int(n))


def perm_product(wires: np.ndarray, idp: np.ndarray, sigma: np.ndarray, beta: np.ndarray, gamma: np.ndarray) -> np.ndarray:
    """dispatcher2.rs:329-345; wires/idp/sigma: [n_types, n, 4] Montgomery Fr"""
    n_types, n = wires.shape[0], wires.shape[1]
    out = np.zeros((n, 4), dtype=np.uint64)
    args = [np.ascontiguousarray(a, dtype=np.uint64) for a in (wires, idp, sigma, beta, gamma)]
    rc = lib().orc_perm_product(_ptr(args[0]), _ptr(args[1]), _ptr(args[2]), n_types, n, _ptr(args[3]), _ptr(args[4]), _ptr(out))
    if rc != 0:
        raise ZeroDivisionError("zero denominator in the permutation product")
    return out


def quotient_evals(selectors, sigmas, wires, perm, pub_input, k, alpha, beta, gamma, n: int) -> np.ndarray:
    """dispatcher2.rs:363-504; selectors [13, m, 4], sigmas / wires [5, m, 4], perm / pub_input [m, 4], k [5, 4]"""
    a = [np.ascontiguousarray(x, dtype=np.uint64) for x in (selectors, sigmas, wires, perm, pub_input, k, alpha, beta, gamma)]
    m = a[3].shape[0]
    out = np.zeros((m, 4), dtype=np.uint64)
    lib().orc_quotient_evals(*[_ptr(x) for x in a], n, m, _ptr(out))
    return out


def poly_eval(coeffs: np.ndarray, point: np.ndarray) -> np.ndarray:
    """DensePolynomial::evaluate (dispatcher2.rs:535-548)"""
    c, z = np.ascontiguousarray(coeffs, dtype=np.uint64), np.ascontiguousarray(point, dtype=np.uint64)
    out = np.zeros(4, dtype=np.uint64)
    lib().orc_poly_eval(_ptr(c), c.shape[0], _ptr(z), _ptr(out))
    return out


def poly_lincomb(polys, coeffs: np.ndarray, out_len: int | None = None) -> np.ndarray:
    """sum_k coeffs[k] * polys[k], shorter polynomials zero-extended (dispatcher2.rs:566-649)"""
    ps = [np.ascontiguousarray(x, dtype=np.uint64) for x in polys]
    cf = np.ascontiguousarray(coeffs, dtype=np.uint64)
    lens = np.array([x.shape[0] for x in ps], dtype=np.uint64)
    n_out = int(lens.max()) if out_len is None else out_len
    ptrs = (C.c_void_p * len(ps))(*[x.ctypes.data for x in ps])
    out = np.zeros((n_out, 4), dtype=np.uint64)
    lib().orc_poly_lincomb(C.cast(ptrs, C.c_void_p), _ptr(lens), _ptr(cf), len(ps), _ptr(out), n_out)
    return out


def poly_div_linear(coeffs: np.ndarray, point: np.ndarray) -> np.ndarray:
    """quotient of p(X) / (X - point): the witness polynomial of dispatcher2.rs:651-666"""
    c, z = np.ascontiguousarray(coeffs, dtype=np.uint64), np.ascontiguousarray(point, dtype=np.uint64)
    out = np.zeros((max(c.shape[0] - 1, 0), 4), dtype=np.uint64)
    lib().orc_poly_div_linear(_ptr(c), c.shape[0], _ptr(z), _ptr(out))
    return out


def gen_srs(tau_canonical: np.ndarray, n: int) -> np.ndarray:
    """[tau^i] G, i < n, as raw GroupAffine structs (tests only: the trapdoor is known)"""
    t = np.ascontiguousarray(tau_canonical, dtype=np.uint64)
    out = np.zeros((n, 104), dtype=np.uint8)
    lib().orc_gen_srs(_ptr(t), n, _ptr(out))
    return out


def g1_mul(aff104: np.ndarray, k_canonical: np.ndarray) -> np.ndarray:
    out = np.zeros(104, dtype=np.uint8)
    lib().orc_g1_mul(_ptr(np.ascontiguousarray(aff104, dtype=np.uint8)), _ptr(np.ascontiguousarray(k_canonical, dtype=np.uint64)), _ptr(out))
    return out


def affine_to_jacobian(aff104: np.ndarray) -> np.ndarray:
    """raw GroupAffine -> raw GroupProjective with z = 1 (identity: (0, 1, 0))"""
    a = np.ascontiguousarray(aff104, dtype=np.uint8)
    out = np.zeros(144, dtype=np.uint8)
    out[:96] = a[:96]
    if a[96]:
        out[:96] = 0
        out[48:96] = _FQ_ONE
    else:
        out[96:144] = _FQ_ONE
    return out


_FQ_ONE = np.array([0x760900000002fffd, 0xebf4000bc40c0002, 0x5f48985753c758ba, 0x77ce585370525745, 0x5c071a97a256ec6d,
                    0x15f65ec3fa80e493], dtype=np.uint64).view(np.uint8)


def g1_compress(bases104: np.ndarray) -> np.ndarray:
    """[n, 104] raw GroupAffine -> [n, 48] ark-serialize compressed"""
    b = np.ascontiguousarray(bases104, dtype=np.uint8).reshape(-1, 104)
    out = np.zeros((b.shape[0], 48), dtype=np.uint8)
    for k in range(b.shape[0]):
        lib().orc_g1_compress(b[k].ctypes.data, out[k].ctypes.data)
    return out


def g1_decompress(comp48: np.ndarray, check_subgroup: bool = True):
    """[n, 48] -> ([n, 104], rc list); rc != 0 marks an invalid encoding (see orc_g1_decompress)"""
    c = np.ascontiguousarray(comp48, dtype=np.uint8).reshape(-1, 48)
    out = np.zeros((c.shape[0], 104), dtype=np.uint8)
    rcs = [lib().orc_g1_decompress(c[k].ctypes.data, out[k].ctypes.data, int(check_subgroup)) for k in range(c.shape[0])]
    return out, rcs


def g1_point_outside_subgroup() -> np.ndarray:
    out = np.zeros(48, dtype=np.uint8)
    assert lib().orc_g1_point_outside_subgroup(out.ctypes.data) == 0
    return out


def vec_op(op: str, a: np.ndarray, b: np.ndarray | None = None) -> np.ndarray:
    """elementwise Fr add / sub / mul / inv over [n, 4] Montgomery arrays (test-instance construction)"""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = a if b is None else np.ascontiguousarray(b, dtype=np.uint64)
    out = np.empty_like(a)
    lib().orc_fr_vec_op(_ptr(a), _ptr(b), _ptr(out), a.shape[0], {"add": 0, "sub": 1, "mul": 2, "inv": 3}[op])
    return out


def into_repr(x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.uint64)
    out = np.empty_like(x)
    lib().orc_fr_into_repr(_ptr(x), _ptr(out), x.shape[0])
    return out


def from_repr(x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.uint64)
    out = np.empty_like(x)
    lib().orc_fr_from_repr(_ptr(x), _ptr(out), x.shape[0])
    return out


def msm(bases: np.ndarray, scalars: np.ndarray) -> np.ndarray:
    n = min(bases.shape[0], scalars.shape[0])
    bases = np.ascontiguousarray(bases[:n])
    scalars = np.ascontiguousarray(scalars[:n], dtype=np.uint64)
    out = np.zeros(144, dtype=np.uint8)
    lib().orc_msm(_ptr(bases), _ptr(scalars), n, _ptr(out))
    return out


def commit(bases: np.ndarray, fr_mont: np.ndarray) -> np.ndarray:
    bases = np.ascontiguousarray(bases)
    fr_mont = np.ascontiguousarray(fr_mont, dtype=np.uint64)
    out = np.zeros(144, dtype=np.uint8)
    lib().orc_commit(_ptr(bases), bases.shape[0], _ptr(fr_mont), fr_mont.shape[0], _ptr(out))
    return out


def normalize(jac144: np.ndarray) -> np.ndarray:
    jac144 = np.ascontiguousarray(jac144, dtype=np.uint8)
    out = np.zeros(104, dtype=np.uint8)
    lib().orc_g1_normalize(_ptr(jac144), _ptr(out))
    return out


def g1_add(a144: np.ndarray, b144: np.ndarray) -> np.ndarray:
    out = np.zeros(144, dtype=np.uint8)
    lib().orc_g1_add(_ptr(np.ascontiguousarray(a144)), _ptr(np.ascontiguousarray(b144)), _ptr(out))
    return out
