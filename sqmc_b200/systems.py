"""Host-side system set-up: the tables the Fortran driver hands to the library.

In the drop-in deployment these tables already exist in the reference's module
globals (``integrals``/``combine_2`` in chemistry.f90, ``k_vectors`` in heg.f90 /
hubbard.f90) and are passed through the C ABI as they are.  This module rebuilds
them in Python/numpy for tests and the benchmark, following the reference's
set-up routines (file:line cited per function, paths relative to
/root/reference/src).  It is host-side one-off set-up, not the hot path.
"""
import math
import re

import numpy as np

# D2h (and its subgroups c1/cs/c2v/c2h) product table, Molpro irrep numbering:
# product(i,j) = ((i-1) xor (j-1)) + 1  (chemistry.f90:7250-7283)


def irrep_product(i, j):
    return ((i - 1) ^ (j - 1)) + 1


class ChemSystem:
    """chem: FCIDUMP + orbital reorder (chemistry.f90:383-398, 538-869, 8921-9022, 9378-9442)."""

    def __init__(self, fcidump, nelec=None, nup=None, orbital_symmetries=None, time_sym=False, z=1, hf_up=None, hf_dn=None):
        header, body = _read_fcidump(fcidump)
        self.norb = norb = _check_norb(int(header["NORB"]))
        self.nelec = int(header["NELEC"]) if nelec is None else nelec
        ms2 = int(header.get("MS2", 0))
        self.nup = (self.nelec + ms2) // 2 if nup is None else nup
        self.ndn = self.nelec - self.nup
        self.time_sym, self.z = bool(time_sym), int(z)
        sym = header.get("ORBSYM") if orbital_symmetries is None else list(orbital_symmetries)
        self.orbital_symmetries_fcidump = np.array(sym if sym else [1] * norb, dtype=np.int32)
        n1 = norb + 1
        # combine_2 initial (chemistry.f90:383-394), 1-based -> index [i-1, j-1]
        c2 = np.zeros((n1, n1), dtype=np.int64)
        for i in range(1, norb + 1):
            for j in range(1, norb + 1):
                c2[i - 1, j - 1] = (i * (i - 1)) // 2 + j if i > j else (j * (j - 1)) // 2 + i
        c2[n1 - 1, n1 - 1] = (n1 * norb) // 2 + n1
        self._c2 = c2
        nint = self._index(n1, n1, n1, n1)
        integrals = np.zeros(nint)
        for v, p, q, r, s in body:  # chemistry.f90:665-682
            p, q, r, s = (x if x != 0 else n1 for x in (p, q, r, s))
            if abs(v) > 1.0e-9:
                integrals[self._index(p, q, r, s) - 1] = v
        self.integrals = integrals
        # HF det: first nup/ndn orbitals unless given (chemistry.f90:694-702)
        if hf_up is None:
            hf_up = (1 << self.nup) - 1
            hf_dn = (1 << self.ndn) - 1
        # sort_integrals (chemistry.f90:8921-9022)
        oe = self._orbital_energies(hf_up, hf_dn)
        tmp = oe.copy()
        for i in range(norb):
            if (hf_up >> i) & 1:
                tmp[i] = tmp[i] - 1.0e9
            if (hf_dn >> i) & 1:
                tmp[i] = tmp[i] - 1.0e9
        order = np.zeros(n1, dtype=np.int64)
        inv = np.zeros(n1, dtype=np.int64)
        order[norb] = n1
        inv[norb] = n1
        for i in range(1, norb + 1):
            mn = tmp.min()
            for j in range(1, norb + 1):
                if tmp[j - 1] == mn:
                    order[i - 1] = j
                    inv[j - 1] = i
                    tmp[j - 1] = 1.0e99
                    break
        self.orb_order, self.orb_order_inv = order, inv
        self.orbital_symmetries = self.orbital_symmetries_fcidump[order[:norb] - 1].copy()
        self.orbital_energies = oe[order[:norb] - 1].copy()
        nu = nd = 0
        for i in range(norb):
            if (hf_up >> i) & 1:
                nu |= 1 << int(inv[i] - 1)
            if (hf_dn >> i) & 1:
                nd |= 1 << int(inv[i] - 1)
        if self.time_sym and nd < nu:
            nu, nd = nd, nu
        self.hf_up, self.hf_dn = nu, nd
        # combine_2 remap (chemistry.f90:855-866)
        for i in range(1, norb + 1):
            a = int(order[i - 1])
            for j in range(1, norb + 1):
                b = int(order[j - 1])
                c2[i - 1, j - 1] = (a * (a - 1)) // 2 + b if a > b else (b * (b - 1)) // 2 + a
        self.combine_2 = np.asfortranarray(c2.astype(np.int32))  # (norb+1)x(norb+1), column-major for the C ABI
        self.enuc = float(integrals[self._index(n1, n1, n1, n1) - 1])

    def _index(self, i, j, k, l):  # chemistry.f90:9106-9134
        a = int(self._c2[i - 1, j - 1])
        b = int(self._c2[k - 1, l - 1])
        return (a * (a - 1)) // 2 + b if a > b else (b * (b - 1)) // 2 + a

    def integral(self, p, q, r, s):
        return self.integrals[self._index(p, q, r, s) - 1]

    def _orbital_energies(self, hf_up, hf_dn):  # chemistry.f90:9378-9442
        norb, n1 = self.norb, self.norb + 1
        oe = np.zeros(norb)
        up = [(hf_up >> k) & 1 for k in range(norb)]
        dn = [(hf_dn >> k) & 1 for k in range(norb)]
        for i in range(1, norb + 1):
            e = self.integral(i, i, n1, n1)
            ex = 0.0
            di = 0.0
            for j in range(1, norb + 1):
                if j != i and up[j - 1]:
                    ex = ex - self.integral(i, j, j, i)
                if j != i and dn[j - 1]:
                    ex = ex - self.integral(i, j, j, i)
            for j in range(1, norb + 1):
                if j != i and up[j - 1]:
                    di = di + self.integral(i, i, j, j)
            for j in range(1, norb + 1):
                if dn[j - 1]:
                    di = di + self.integral(i, i, j, j)
            for j in range(1, norb + 1):
                if j != i and dn[j - 1]:
                    di = di + self.integral(i, i, j, j)
            for j in range(1, norb + 1):
                if up[j - 1]:
                    di = di + self.integral(i, i, j, j)
            oe[i - 1] = e + 0.5 * (ex + di)
        return oe

    # dense helper tables in the reordered orbital numbering (used by spaces.py)
    def jk_tables(self):
        norb, n1 = self.norb, self.norb + 1
        h = np.array([self.integral(i, i, n1, n1) for i in range(1, norb + 1)])
        J = np.array([[self.integral(i, i, j, j) for j in range(1, norb + 1)] for i in range(1, norb + 1)])
        K = np.array([[self.integral(i, j, j, i) for j in range(1, norb + 1)] for i in range(1, norb + 1)])
        return h, J, K


def _check_norb(norb):
    """a determinant string is two 64-bit words holding a value below 2^127 (types.f90:44): 1..127 orbitals"""
    if not 1 <= norb <= 127:
        raise ValueError("norb=%d outside 1..127: determinant strings hold at most 127 orbitals" % norb)
    return norb


def _read_fcidump(path):
    with open(path) as f:
        lines = f.read().splitlines()
    # header = everything up to and including the line with &END or '/'
    end = None
    for k, ln in enumerate(lines):
        u = ln.upper()
        if "&END" in u or u.strip() == "/" or u.strip().endswith("/"):
            end = k
            break
    if end is None:
        raise ValueError("FCIDUMP: no &END line")
    text = " ".join(lines[:end + 1])
    header = {}
    for key in ("NORB", "NELEC", "MS2", "ISYM"):
        m = re.search(key + r"\s*=\s*(-?\d+)", text, re.I)
        if m:
            header[key] = int(m.group(1))
    m = re.search(r"ORBSYM\s*=\s*([\d,\s]+)", text, re.I)
    if m:
        header["ORBSYM"] = [int(x) for x in m.group(1).replace(",", " ").split()]
    body = []
    for ln in lines[end + 1:]:
        t = ln.split()
        if len(t) < 5:
            continue
        body.append((float(t[0].replace("D", "E").replace("d", "e")), int(t[1]), int(t[2]), int(t[3]), int(t[4])))
    return header, body


class HegSystem:
    """heg: k-vectors inside the cutoff sphere, ordered by the reference's shell sort
    (heg.f90:173-240, 643-749; generic_sort.f90:554-592)."""

    def __init__(self, n_dim, r_s, nelec, nup, cutoff_radius):
        EPS = 1.0e-15
        self.n_dim, self.r_s, self.nelec, self.nup, self.ndn = n_dim, r_s, nelec, nup, nelec - nup
        density = 1.0 / (math.pi * r_s ** 2) if n_dim == 2 else 3.0 / (4.0 * math.pi * r_s ** 3)
        self.length_cell = (nelec / density) ** (1.0 / n_dim)
        n_max = int(cutoff_radius + EPS)
        values = [2 * math.pi / self.length_cell * i for i in range(-n_max, n_max + 1)]
        kv = []
        if n_dim == 3:
            for i in range(-n_max, n_max + 1):
                for j in range(-n_max, n_max + 1):
                    for k in range(-n_max, n_max + 1):
                        kv.append([values[i + n_max], values[j + n_max], values[k + n_max]])
        else:
            for i in range(-n_max, n_max + 1):
                for j in range(-n_max, n_max + 1):
                    kv.append([values[i + n_max], values[j + n_max]])

        def s2(v):
            s = 0.0
            for x in v:
                s += x * x
            return s

        ntot = len(kv)
        inc = ntot // 2
        while inc > 0:  # shell sort, 1-based indices as in the Fortran
            for i in range(inc + 1, ntot + 1):
                j = i
                temp = kv[i - 1]
                while j >= inc + 1:
                    if s2(kv[j - inc - 1]) <= s2(temp):
                        break
                    kv[j - 1] = kv[j - inc - 1]
                    j -= inc
                kv[j - 1] = temp
            inc = 1 if inc == 2 else inc * 5 // 11
        norb = 0
        for v in kv:
            if math.sqrt(s2(v)) > 2 * math.pi / self.length_cell * cutoff_radius + EPS:
                break
            norb += 1
        self.norb = _check_norb(norb)
        self.k_vectors = np.array(kv[:norb], dtype=np.float64)  # (norb, n_dim) C-order == (n_dim, norb) column-major
        self.hf_up = (1 << nup) - 1
        self.hf_dn = (1 << self.ndn) - 1


class HubbardKSystem:
    """hubbardk: momentum orbitals sorted by energy (hubbard.f90:2179-2290)."""

    def __init__(self, l_x, l_y, t, U, nup, ndn):
        self.l_x, self.l_y, self.t, self.U, self.nup, self.ndn = l_x, l_y, t, U, nup, ndn
        ns = l_x * l_y
        self.norb = _check_norb(ns)
        kv = np.zeros((ns, 2), dtype=np.int64)
        for i in range(1, l_x + 1):
            for j in range(1, l_y + 1):
                kv[l_y * (i - 1) + j - 1] = (-l_x + 2 * i, -l_y + 2 * j)
        if l_x % 2 == 1:
            kv[:, 0] -= 1
        if l_y % 2 == 1:
            kv[:, 1] -= 1
        ke = np.zeros(ns)
        for o in range(ns):
            if l_y == 1:
                ke[o] = -2.0 * t * (math.cos(math.pi * kv[o, 0] / float(l_x)))
            elif l_x == 1:
                ke[o] = -2.0 * t * (math.cos(math.pi * kv[o, 1] / float(l_y)))
            else:
                ke[o] = -2.0 * t * (math.cos(math.pi * kv[o, 0] / float(l_x)) + math.cos(math.pi * kv[o, 1] / float(l_y)))
        tmp = ke.copy()
        order = []
        for _ in range(ns):
            mn = tmp.min()
            for j in range(ns):
                if tmp[j] == mn:
                    tmp[j] = tmp.max() + 1.0
                    order.append(j)
                    break
        self.k_vectors = np.ascontiguousarray(kv[order].astype(np.int32))  # (nsites, 2) C-order == (2, nsites) column-major
        self.k_energies = ke[order].copy()
        self.ubyn = U / float(ns)

    def total_momentum(self, up, dn):
        kx = ky = 0
        for o in range(self.norb):
            c = ((up >> o) & 1) + ((dn >> o) & 1)
            kx += c * int(self.k_vectors[o, 0])
            ky += c * int(self.k_vectors[o, 1])
        return kx % (2 * self.l_x), ky % (2 * self.l_y)
