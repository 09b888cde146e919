"""Reference file formats on either side of the hot path (SURVEY.md section 8(f) items 2 and 3).

  * `wf_eps_var=<eps>`  -- the variational wavefunction checkpoint perform_hci writes / reads
    (hci.f90:194-231 read, :601-625 write): a Fortran *sequential unformatted* file with five records
        ndets (default integer, 4 B) | dets_up(1:ndets) integer(16) | dets_dn(1:ndets) integer(16) |
        wts(1:ndets,1:n_states) real(8), column-major | energy(1:n_states) real(8)
    written by gfortran (src/Makefile:18): every record is framed by 4-byte little-endian length markers;
    records longer than 2 147 483 639 bytes are split into subrecords whose leading marker is negative when
    another subrecord follows and whose trailing marker is negative when one precedes.
  * `dtm_projector` text file -- the deterministic-space Hamiltonian walk dumps / loads
    (do_walk.f90:964-1013 write, :883-945 read), list-directed:
        n_imp  nnz_upper  dtm_energy  <free text>
        H_nonzero_elements(1:n_imp)                       (one line, i8 fields)
        i  orb_up(1:nup-ncore)  orb_dn(1:ndn-ncore)       (n_imp lines, 1-based orbitals, core orbitals removed)
        H_index  H_value                                  (nnz_upper lines; H itself, the reader applies -tau)

No Fortran compiler exists in the build image, so these layouts are restated from the read/write statements and
gfortran's documented record framing: "parity unpinned by the reference" (no sample file ships with it); the tests
pin the byte layout against hand-assembled records.  Host-side numpy only; nothing here touches the GPU.
"""
import struct

import numpy as np

MAX_SUBRECORD = 2147483639  # gfortran's default -fmax-subrecord-length


# ----------------------------------------------------------------------------- unformatted sequential records
def _write_record(f, payload, max_sub=MAX_SUBRECORD):
    payload = memoryview(payload).cast("B")
    n = len(payload)
    if n == 0:
        f.write(struct.pack("<ii", 0, 0))
        return
    off, first = 0, True
    while off < n:
        m = min(max_sub, n - off)
        more = off + m < n
        f.write(struct.pack("<i", -m if more else m))        # leading marker: negative = continued
        f.write(payload[off:off + m])
        f.write(struct.pack("<i", m if first else -m))        # trailing marker: negative = has a predecessor
        off += m
        first = False


def _read_record(f):
    chunks = []
    while True:
        head = f.read(4)
        if len(head) == 0 and not chunks:
            return None
        if len(head) != 4:
            raise ValueError("truncated record marker")
        (m,) = struct.unpack("<i", head)
        size = abs(m)
        data = f.read(size)
        if len(data) != size:
            raise ValueError("truncated record: wanted %d bytes, got %d" % (size, len(data)))
        tail = f.read(4)
        if len(tail) != 4 or abs(struct.unpack("<i", tail)[0]) != size:
            raise ValueError("record markers disagree")
        chunks.append(data)
        if m >= 0:
            break
    return b"".join(chunks)


# ----------------------------------------------------------------------------- wf_eps_var=...
def wf_filename(eps_var):
    """'wf_eps_var=' // es7.2e1 of eps_var (hci.f90:196-197); exponents that need two digits overflow the field."""
    m, e = ("%.2E" % float(eps_var)).split("E")
    e = int(e)
    if abs(e) > 9:
        return "wf_eps_var=" + "*" * 7
    return "wf_eps_var=%sE%s%d" % (m, "-" if e < 0 else "+", abs(e))


def write_wf(path, up, dn, wts, energies, max_sub=MAX_SUBRECORD):
    """up, dn: (n,2) uint64 (low word first = the little-endian integer(16)); wts: (n, n_states); energies: (n_states,)"""
    up = np.ascontiguousarray(up, dtype="<u8").reshape(-1, 2)
    dn = np.ascontiguousarray(dn, dtype="<u8").reshape(-1, 2)
    n = len(up)
    wts = np.asarray(wts, dtype="<f8").reshape(n, -1)
    energies = np.ascontiguousarray(energies, dtype="<f8").reshape(-1)
    if len(dn) != n or wts.shape[1] != len(energies):
        raise ValueError("write_wf: inconsistent shapes")
    if n >= 2 ** 31:
        raise ValueError("write_wf: ndets does not fit the reference's default integer")
    with open(path, "wb") as f:
        _write_record(f, struct.pack("<i", n), max_sub)
        _write_record(f, up.tobytes(), max_sub)
        _write_record(f, dn.tobytes(), max_sub)
        _write_record(f, np.asfortranarray(wts).tobytes(order="F"), max_sub)
        _write_record(f, energies.tobytes(), max_sub)


def read_wf(path):
    """-> dict(up (n,2) uint64, dn, wts (n, n_states), energies (n_states,)); n_states follows from the record sizes"""
    with open(path, "rb") as f:
        rec = [_read_record(f) for _ in range(5)]
    if any(r is None for r in rec):
        raise ValueError("read_wf: fewer than five records")
    (n,) = struct.unpack("<i", rec[0][:4])
    if len(rec[1]) != 16 * n or len(rec[2]) != 16 * n:
        raise ValueError("read_wf: determinant records do not hold ndets integer(16) values")
    n_states = len(rec[4]) // 8
    if n_states < 1 or len(rec[3]) != 8 * n * n_states:
        raise ValueError("read_wf: weight record does not match ndets x n_states")
    up = np.frombuffer(rec[1], dtype="<u8").reshape(n, 2).copy()
    dn = np.frombuffer(rec[2], dtype="<u8").reshape(n, 2).copy()
    wts = np.frombuffer(rec[3], dtype="<f8").reshape((n, n_states), order="F").copy()
    return dict(up=up, dn=dn, wts=wts, energies=np.frombuffer(rec[4], dtype="<f8").copy())


# ----------------------------------------------------------------------------- dtm_projector text file
def _orbitals(word_pair, n_core_orb):
    v = int(word_pair[0]) | (int(word_pair[1]) << 64)
    out = []
    o = 0
    while v:
        if v & 1 and o >= n_core_orb:
            out.append(o + 1 - n_core_orb)
        v >>= 1
        o += 1
    return out


def write_dtm_projector(path, up, dn, counts, indices, values, dtm_energy=0.0, n_core_orb=0):
    """values = H (NOT -tau*H): do_walk.f90:1007 writes -minus_tau_H_values/tau.  counts/indices as export_upper returns them."""
    up = np.asarray(up, dtype=np.uint64).reshape(-1, 2)
    dn = np.asarray(dn, dtype=np.uint64).reshape(-1, 2)
    counts = np.asarray(counts, dtype=np.int64)
    indices = np.asarray(indices, dtype=np.int64)
    values = np.asarray(values, dtype=np.float64)
    n = len(up)
    if len(counts) != n or counts.sum() != len(indices) or len(indices) != len(values):
        raise ValueError("write_dtm_projector: inconsistent sizes")
    with open(path, "w") as f:
        f.write(" %11d %11d %25.16E  number of deterministic dets, number of nonzero deterministic Hamiltonian elements, "
                "ground state energy within deterministic space\n" % (n, len(indices), dtm_energy))
        f.write("".join("%8d" % c for c in counts) + "\n")
        for i in range(n):
            orbs = _orbitals(up[i], n_core_orb) + _orbitals(dn[i], n_core_orb)
            f.write(" %11d" % (i + 1) + "".join(" %11d" % o for o in orbs) + "\n")
        for k in range(len(indices)):
            f.write(" %19d %25.16E\n" % (indices[k], values[k]))


def read_dtm_projector(path, nup, ndn, n_core_orb=0):
    """-> dict(up, dn (n,2) uint64, counts, indices (1-based), values = H, dtm_energy or None).  Mirrors do_walk.f90:897-945:
    list-directed reads, determinant lines carry their own index, core orbitals are re-inserted."""
    with open(path) as f:
        head = f.readline().replace(",", " ").split()
        n, nnz = int(head[0]), int(head[1])
        try:
            energy = float(head[2].replace("D", "E").replace("d", "E"))
        except (IndexError, ValueError):
            energy = None
        counts = []
        while len(counts) < n:                       # read(57,*) array: continues over as many lines as needed
            counts += [int(t) for t in f.readline().replace(",", " ").split()]
        counts = np.array(counts[:n], dtype=np.int64)
        up = np.zeros((n, 2), dtype=np.uint64)
        dn = np.zeros((n, 2), dtype=np.uint64)
        core = (1 << n_core_orb) - 1
        nu, nd = nup - n_core_orb, ndn - n_core_orb
        for _ in range(n):
            t = [int(x) for x in f.readline().replace(",", " ").split()]
            if len(t) != 1 + nu + nd:
                raise ValueError("read_dtm_projector: determinant line with %d fields, expected %d" % (len(t), 1 + nu + nd))
            ind = t[0] - 1
            a, b = core, core
            for o in t[1:1 + nu]:
                a |= 1 << (o + n_core_orb - 1)
            for o in t[1 + nu:]:
                b |= 1 << (o + n_core_orb - 1)
            up[ind] = (a & 0xFFFFFFFFFFFFFFFF, a >> 64)
            dn[ind] = (b & 0xFFFFFFFFFFFFFFFF, b >> 64)
        indices = np.zeros(nnz, dtype=np.int64)
        values = np.zeros(nnz)
        for k in range(nnz):
            t = f.readline().replace(",", " ").split()
            indices[k] = int(t[0])
            values[k] = float(t[1].replace("D", "E").replace("d", "E"))
    if counts.sum() != nnz:
        raise ValueError("read_dtm_projector: per-row counts sum to %d, header says %d" % (counts.sum(), nnz))
    return dict(up=up, dn=dn, counts=counts, indices=indices, values=values, dtm_energy=energy)


# ----------------------------------------------------------------------------- FCIDUMP
def write_fcidump(path, h, eri, ecore, nelec, ms2=0, orbsym=None, isym=1, tol=1.0e-12):
    """Write a molecular FCIDUMP: the header (NORB, NELEC, MS2, ORBSYM, ISYM), then the unique entries with |v| > tol in the
    usual order -- (pq|rs) with p >= q, r >= s, pq >= rs, then h_pq with p >= q as `v p q 0 0`, then the core energy as
    `v 0 0 0 0`.  h: (norb, norb) symmetric, eri: (norb,)*4 chemists' (pq|rs) with the 8-fold symmetry; orbitals 1-based
    in the file.  Values are written with 17 significant digits, so a read returns them bit for bit."""
    norb = h.shape[0]
    orbsym = [1] * norb if orbsym is None else [int(x) for x in orbsym]
    lines = [" &FCI NORB=%d,NELEC=%d,MS2=%d," % (norb, nelec, ms2), "  ORBSYM=" + "".join("%d," % x for x in orbsym),
             "  ISYM=%d," % isym, " &END"]
    for p in range(norb):
        for q in range(p + 1):
            pq = p * (p + 1) // 2 + q
            for r in range(p + 1):
                for s in range(r + 1):
                    if r * (r + 1) // 2 + s > pq:
                        break
                    v = eri[p, q, r, s]
                    if abs(v) > tol:
                        lines.append("%.17g %d %d %d %d" % (v, p + 1, q + 1, r + 1, s + 1))
    for p in range(norb):
        for q in range(p + 1):
            if abs(h[p, q]) > tol:
                lines.append("%.17g %d %d 0 0" % (h[p, q], p + 1, q + 1))
    lines.append("%.17g 0 0 0 0" % ecore)
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
