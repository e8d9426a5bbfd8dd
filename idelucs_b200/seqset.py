"""Device-resident packed sequence sets (K1).

A ``SeqSet`` is what the reference re-creates from the FASTA file on every pass
(idelucs/utils.py:229-261): here the file is parsed once, the ASCII bytes are copied to
the GPU once and packed there to 2 bits per base + a 1-bit reset mask.
"""
import numpy as np
import torch

from . import _lib

CHUNK = 64


def _check_header(header: str):
    """idelucs/utils.py:37-40"""
    if len(header) > 0 and (header[0] in (">", "#") or header[0].isspace()):
        raise ValueError("Bad character in sequence header")
    if "\t" in header:
        raise ValueError("tab included in header")


def read_fasta_raw(fname):
    """Record iteration of idelucs/utils.py:229-261 (kmersFasta): '#' lines skipped, id =
    header line minus '>' and minus its last byte, sequence lines ``strip()``-ped and joined,
    a record is flushed only while the running id is non-empty, the last record always.
    Returns (names, [bytes]) — alphabet handling happens on the GPU (idl_pack)."""
    names, seqs, lines = [], [], []
    seq_id = ""
    with open(fname, "rb") as fh:
        for line in fh:
            if line.startswith(b"#"):
                continue
            if line.startswith(b">"):
                if seq_id != "":
                    names.append(seq_id)
                    seqs.append(b"".join(lines))
                    lines = []
                seq_id = line[1:-1].decode()
            else:
                lines.append(line.strip())
    names.append(seq_id)
    seqs.append(b"".join(lines))
    return names, seqs


def read_fasta_native(fname, pinned=None):
    """The same record iteration by the native scanner (idl_fasta_scan / idl_fasta_extract): the file is mapped
    once and the stripped sequence lines are concatenated into one flat (pinned, when a GPU is present) uint8
    tensor.  Returns (names, flat uint8 tensor, byte_off int64[n+1])."""
    import ctypes
    import os
    lib = _lib.load()
    if pinned is None:
        pinned = torch.cuda.is_available()
    size = os.path.getsize(fname)
    # the file image is the page cache itself (read-only mapping): no copy before the scan
    bnp = np.memmap(fname, dtype=np.uint8, mode="r") if size else np.zeros(1, np.uint8)
    buf_ptr = ctypes.c_void_p(bnp.ctypes.data)
    n_rec, n_seq = ctypes.c_int64(0), ctypes.c_int64(0)
    _lib.check(lib.idl_fasta_scan(buf_ptr, size, ctypes.byref(n_rec), ctypes.byref(n_seq)))
    n = n_rec.value
    flat = torch.empty(max(n_seq.value, 1), dtype=torch.uint8, pin_memory=bool(pinned))
    byte_off = np.zeros(n + 1, np.int64)
    hdr_off, hdr_len = np.zeros(n, np.int64), np.zeros(n, np.int64)
    _lib.check(lib.idl_fasta_extract(buf_ptr, size, n, _lib.ptr(flat), n_seq.value, byte_off.ctypes.data_as(ctypes.c_void_p),
                                     hdr_off.ctypes.data_as(ctypes.c_void_p), hdr_len.ctypes.data_as(ctypes.c_void_p)))
    mv = memoryview(bnp)
    names = [bytes(mv[o:o + l]).decode() for o, l in zip(hdr_off.tolist(), hdr_len.tolist())]
    return names, flat[: n_seq.value], byte_off


class SeqSet(object):
    """n sequences packed on one GPU.  Tensors: codes (int32 words, 2 bit/base), nmask
    (int32 words, 1 bit/base), chunk_off (int64[n+1]), len (int32[n])."""

    def __init__(self):
        self.names = []
        self.n = 0
        self.lengths = np.zeros(0, np.int64)
        self.codes = self.nmask = self.chunk_off = self.len = None
        self.device = None

    @property
    def total_bases(self):
        return int(self.lengths.sum())

    @classmethod
    def from_ascii(cls, ascii_u8, byte_off, names=None, alphabet="check", device=None, validate=True):
        """ascii_u8: 1-D uint8 array/tensor (host, ideally pinned, or already on the device)
        holding the concatenated sequences; byte_off: int64[n+1] numpy."""
        lib = _lib.load()
        device = torch.device(device if device is not None else "cuda")
        self = cls()
        byte_off = np.ascontiguousarray(byte_off, dtype=np.int64)
        n = byte_off.size - 1
        lengths = np.diff(byte_off)
        if n > 0 and lengths.max() > 0x7fffffff:
            raise ValueError("sequence longer than 2^31-1 bases")
        chunk_off = np.zeros(n + 1, np.int64)
        np.cumsum((lengths + CHUNK - 1) // CHUNK, out=chunk_off[1:])
        total_chunks = int(chunk_off[-1])
        self.n, self.lengths = n, lengths
        self.names = list(names) if names is not None else [str(i) for i in range(n)]
        self.device = device
        if isinstance(ascii_u8, np.ndarray):
            ascii_u8 = torch.from_numpy(np.ascontiguousarray(ascii_u8, dtype=np.uint8))
        d_ascii = ascii_u8.to(device, non_blocking=True) if ascii_u8.numel() else torch.zeros(1, dtype=torch.uint8, device=device)
        d_byte_off = torch.from_numpy(byte_off).to(device, non_blocking=True)
        self.chunk_off = torch.from_numpy(chunk_off).to(device, non_blocking=True)
        self.codes = torch.empty((total_chunks + 1) * 4, dtype=torch.int32, device=device)
        self.nmask = torch.empty((total_chunks + 1) * 2, dtype=torch.int32, device=device)
        self.len = torch.empty(max(n, 1), dtype=torch.int32, device=device)
        bad = torch.full((max(n, 1),), -1, dtype=torch.int64, device=device)
        with torch.cuda.device(device):
            _lib.check(lib.idl_pack(_lib.ptr(d_ascii), _lib.ptr(d_byte_off), n, 1 if alphabet == "strict" else 0,
                                    int(lengths.max()) if n else 0, _lib.ptr(self.chunk_off), _lib.ptr(self.codes),
                                    _lib.ptr(self.nmask), _lib.ptr(self.len), _lib.ptr(bad), _lib.stream_ptr()))
        self._bad = bad
        self._d_ascii = d_ascii
        if validate:
            self.validate()
        return self

    def validate(self, header_error=None):
        """Raise what check_sequence raises (idelucs/utils.py:37-50), for the first offending
        record in file order.  header_error = (index, exception) of the first bad header.
        Returns the indices of sequences that contain deletable whitespace (the caller
        compacts those on the host and re-packs before errors are final)."""
        bad = self._bad[: self.n].cpu().numpy()
        hit = np.nonzero(bad != -1)[0]
        h_idx = header_error[0] if header_error else self.n + 1
        ws = []
        for i in hit:
            if i >= h_idx:
                break
            v = int(bad[i])
            if (v & 7) == 6:
                if ws:            # an earlier record needs compaction first: decide afterwards
                    return ws
                b0 = int(self.lengths[:i].sum())
                byte = int(self._d_ascii[b0 + (v >> 3)].item())
                raise ValueError("Invalid DNA byte in sequence {}: '{}'".format(self.names[i], chr(byte)))
            ws.append(int(i))
        if ws:
            return ws
        if header_error:
            raise header_error[1]
        return ws

    @classmethod
    def from_sequences(cls, seqs, names=None, alphabet="check", device=None, pinned=False):
        """seqs: iterable of bytes-like.  check_sequence semantics (utils.py:42-50): whitespace
        ' \\t\\n\\r' is deleted, IUPAC/'-' -> N, invalid bytes raise ValueError."""
        seqs = [bytes(s) for s in seqs]
        header_error = None
        if names is not None and alphabet == "check":
            for i, h in enumerate(names):
                try:
                    _check_header(h)
                except ValueError as e:
                    header_error = (i, e)
                    break
        for attempt in range(2):
            lengths = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
            byte_off = np.zeros(len(seqs) + 1, np.int64)
            np.cumsum(lengths, out=byte_off[1:])
            flat = np.frombuffer(b"".join(seqs), dtype=np.uint8)
            t = torch.from_numpy(flat.copy()) if flat.size else torch.zeros(0, dtype=torch.uint8)
            if pinned and flat.size:
                t = t.pin_memory()
            self = cls.from_ascii(t, byte_off, names=names, alphabet=alphabet, device=device, validate=False)
            ws = self.validate(header_error) if alphabet == "check" else []
            if not ws:
                return self
            if attempt == 1:
                raise RuntimeError("whitespace survived compaction")
            for i in ws:  # rare path: the reference deletes these bytes (utils.py:45)
                seqs[i] = seqs[i].translate(None, b" \t\n\r")
        return self

    @classmethod
    def from_fasta(cls, fname, device=None, rows=None):
        """Parse once with the native scanner, one H2D copy of the flat pinned bytes, pack on the device.  Records
        whose sequence lines hold interior whitespace (deleted by check_sequence, utils.py:45) take the host
        compaction path of from_sequences.  rows = (lo, hi): pack only records lo .. hi-1 (one rank's shard)."""
        names, flat, byte_off = read_fasta_native(fname)
        if rows is not None:
            lo, hi = rows
            flat, byte_off, names = flat[int(byte_off[lo]):int(byte_off[hi])], byte_off[lo:hi + 1] - byte_off[lo], names[lo:hi]
        header_error = None
        for i, h in enumerate(names):
            try:
                _check_header(h)
            except ValueError as e:
                header_error = (i, e)
                break
        self = cls.from_ascii(flat, byte_off, names=names, device=device, validate=False)
        if not self.validate(header_error):
            return self
        fl = flat.numpy()
        seqs = [fl[byte_off[i]:byte_off[i + 1]].tobytes() for i in range(len(names))]
        return cls.from_sequences(seqs, names=names, device=device)
