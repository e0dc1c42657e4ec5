"""np.loadtxt feature matrices read straight into device memory: the host streams the file, the device parses it (K8,
mlbp_parse_float_text in csrc/parse.cu).

train.py:589-603 reads the four feature matrices with np.loadtxt(path, dtype=float64); the engine then casts them to fp32, pads
every row to ld elements and uploads them (Model.__init__).  Here each file is read with readinto() into one of two reusable
pinned buffers, cut after its last newline (the tail is carried into the next chunk), copied with a non-blocking copy_ and
parsed on the device straight into the padded plane, while the host reads the next chunk.  The host never holds a matrix.

The result is bit-identical to the np.loadtxt path: every field is converted to the correctly rounded float64 and then rounded
to fp32, and the float64 min / max that set Model.frange and Model.ed_range are taken on the device.  Fields whose rounding the
device leaves open (more than 19 significant digits, rare) are re-read here with float().

Whenever the device does not report a clean file of the expected shape -- a syntax error, a ragged line, a byte outside
the ASCII grammar (a non-ASCII comment, say), a row count other than the vocabulary size -- the file is read with np.loadtxt
instead and goes down the np.loadtxt path unchanged, so an invalid file raises exactly np.loadtxt's exception.
"""
import ctypes
import struct
import time
import warnings

import numpy as np
import torch

# include/mlbp.h MLBP_PARSE_*
STATE_WORDS, W_FIELDS, W_ERROR, W_MIN, W_MAX, W_NAN, W_HARD = 8, 0, 1, 2, 3, 4, 5
TILE_BYTES = 4096
MAX_CHUNK = (1 << 31) - 1
ERROR_KINDS = {1: 'a malformed field', 2: 'a line with another number of fields', 3: 'more rows than expected',
               4: 'a byte outside the ASCII grammar'}
HARD_CAP = 1 << 16            # listed hard fields per file; more send the file to np.loadtxt
DEFAULT_CHUNK_BYTES = 256 << 20
MASK64 = (1 << 64) - 1


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _float_of_bits(b):
    return struct.unpack('<d', struct.pack('<Q', b & MASK64))[0]


def _float_of_key(key):
    """inverse of the kernel's order key: key(b) = b ^ (sign ? ~0 : 1 << 63)"""
    return _float_of_bits(key ^ (1 << 63) if key >> 63 else ~key)


def _last_newline(a):
    """index of the last b'\\n' in the uint8 array a, or -1 (searched from the end in growing windows)"""
    hi, step = len(a), 1 << 16
    while hi > 0:
        lo = max(0, hi - step)
        nz = np.flatnonzero(a[lo:hi] == 10)
        if len(nz):
            return lo + int(nz[-1])
        hi, step = lo, step * 4
    return -1


def first_row_fields(path):
    """number of fields on the first line that has any (what np.loadtxt takes the column count from)"""
    with open(path, 'rb') as f:
        for line in f:
            n = len(line.split(b'#', 1)[0].split())
            if n:
                return n
    return 0


def _field_text(f, offset):
    """the bytes of the field that starts at byte `offset` of the open file f"""
    f.seek(offset)
    out = b''
    while True:
        piece = f.read(4096)
        cut = [i for i, c in enumerate(piece) if c in b' \t\n\r\x0b\x0c#']
        if cut or not piece:
            return out + piece[:cut[0] if cut else len(piece)]
        out += piece


class TextLoader(object):
    """Parses np.loadtxt text files into device planes with one set of reusable buffers."""

    def __init__(self, kernels, chunk_bytes=None):
        self.k = kernels
        self.device = kernels.device
        self.chunk_bytes = int(chunk_bytes or DEFAULT_CHUNK_BYTES)
        assert 1 <= self.chunk_bytes <= MAX_CHUNK // 2
        self.pin = self.device.type == 'cuda'
        self._host = [None, None]                 # the two pinned read buffers
        self._dev = None
        self._ws = None
        self.state = torch.zeros(STATE_WORDS, dtype=torch.int64, device=self.device)
        self.hard = torch.zeros(2 * HARD_CAP, dtype=torch.int64, device=self.device)
        self.stats = {'bytes': 0, 'chunks': 0, 'hard_fields': 0, 'read_seconds': 0.0}

    def _host_buffer(self, j, need):
        if self._host[j] is None or self._host[j].numel() < need:
            self._host[j] = torch.empty(max(need, self.chunk_bytes + 1), dtype=torch.uint8, pin_memory=self.pin)
        return self._host[j]

    def _device_buffers(self, n):
        if self._dev is None or self._dev.numel() < n:
            self._dev = torch.empty(max(n, self.chunk_bytes), dtype=torch.uint8, device=self.device)
            self._ws = torch.empty(-(-self._dev.numel() // TILE_BYTES), dtype=torch.int64, device=self.device)
        return self._dev, self._ws

    def parse(self, path, rows, cols, out, ld_out):
        """Parse the text file `path` of a rows x cols matrix into out[r * ld_out + c] (a contiguous fp32 device tensor).
        Returns (min, max) of the float64 values, or a string saying why the device did not read a clean file of this
        shape (then `out` holds garbage)."""
        n_cols = first_row_fields(path)
        if n_cols != cols:
            return 'its first line has %d fields, not %d' % (n_cols, cols)
        self.k.call('mlbp_zero_words', _ptr(self.state), 2 * STATE_WORDS)
        events = [None, None]
        tail, offset, j = None, 0, 0
        with open(path, 'rb', buffering=0) as f:
            while True:
                if events[j] is not None:
                    events[j].synchronize()       # the copy out of this buffer has finished
                c = 0 if tail is None else len(tail)
                hb = self._host_buffer(j, c + self.chunk_bytes)
                buf = hb.numpy()
                if c:
                    buf[:c] = tail
                t0 = time.perf_counter()
                got = f.readinto(memoryview(buf)[c:c + self.chunk_bytes])
                self.stats['read_seconds'] += time.perf_counter() - t0
                n = c + got
                eof = got == 0
                nl = _last_newline(buf[c:n])      # (the carried tail holds no newline)
                cut = n if eof else (c + nl + 1 if nl >= 0 else 0)   # after the last newline; 0: no complete line yet
                events[j] = None
                if cut > 0:
                    dev, ws = self._device_buffers(cut)
                    dev[:cut].copy_(hb[:cut], non_blocking=True)
                    if self.pin:
                        events[j] = torch.cuda.Event()
                        events[j].record()
                    self.k.call('mlbp_parse_float_text', _ptr(dev), cut, offset, cols, rows, _ptr(out), ld_out,
                                _ptr(self.state), _ptr(self.hard), HARD_CAP, _ptr(ws))
                    self.stats['chunks'] += 1
                offset += cut
                tail = buf[cut:n]                 # (a view: this buffer is not written again before the copy below)
                j ^= 1
                if eof:
                    break
            self.stats['bytes'] += offset
            st = [int(x) & MASK64 for x in self.state.cpu().tolist()]
            if st[W_ERROR]:
                e = ~st[W_ERROR] & MASK64
                return '%s at byte %d' % (ERROR_KINDS.get(e & 7, 'error %d' % (e & 7)), e >> 3)
            if st[W_FIELDS] != rows * cols:
                return '%d fields, not %d x %d' % (st[W_FIELDS], rows, cols)
            n_hard = st[W_HARD]
            if n_hard > HARD_CAP:
                return '%d fields with more than 19 significant digits' % n_hard
            lo = _float_of_key(~st[W_MIN] & MASK64) if st[W_MIN] else None
            hi = _float_of_key(st[W_MAX]) if st[W_MAX] else None
            if n_hard:
                # fields the device could not round from 19 digits: float() on the host, patched into the plane
                pairs = sorted(map(tuple, self.hard[:2 * n_hard].view(-1, 2).cpu().tolist()), key=lambda p: p[1])
                vals = [float(_field_text(f, off)) for off, _ in pairs]
                idx = torch.tensor([(k // cols) * ld_out + k % cols for _, k in pairs], dtype=torch.int64)
                out.view(-1)[idx.to(self.device)] = torch.tensor(np.asarray(vals, dtype=np.float32)).to(self.device)
                lo = min([lo] + vals if lo is not None else vals)
                hi = max([hi] + vals if hi is not None else vals)
                self.stats['hard_fields'] += n_hard
        if st[W_NAN]:                             # np.min / np.max return NaN when there is one
            nan = -float('nan') if st[W_NAN] == 2 else float('nan')
            return nan, nan
        return lo, hi


def model_from_text(cls, paths, V, Vd, kernels, chunk_bytes=None):
    """Model.from_text: the four feature planes of `cls` (engine.Model) parsed on the device (see the module docstring)."""
    ld = (V + 63) // 64 * 64
    loader = TextLoader(kernels, chunk_bytes)
    dev = loader.device
    shapes = {'pmi': (V, V), 'pmi_w1': (V, V), 'ed': (V, Vd), 'ped': (V, Vd)}
    names = ('pmi', 'pmi_w1', 'ed', 'ped')
    planes, ranges, host, why = {}, {}, {}, []
    for name, path in zip(names, paths):
        rows, cols = shapes[name]
        t = torch.zeros((rows, ld if name.startswith('pmi') else cols), dtype=torch.float32, device=dev)
        r = loader.parse(path, rows, cols, t, t.shape[1])
        if not isinstance(r, str):
            planes[name], ranges[name] = t, r
            continue
        if not why:
            warnings.warn('%s: %s; reading it with np.loadtxt' % (path, r), RuntimeWarning, stacklevel=3)
        why.append((path, r))
        host[name] = np.loadtxt(path, dtype=np.float64, ndmin=2)
        if host[name].shape != (rows, cols):
            # not the shape the vocabularies give: the np.loadtxt path for every file, then Model() as before
            arrays = [host[n] if n in host else np.loadtxt(p, dtype=np.float64, ndmin=2) for n, p in zip(names, paths)]
            return cls(*arrays, device=dev)
    m = cls.__new__(cls)
    m.V, m.Vd, m.ld, m.device = V, Vd, ld, dev
    m.load_stats = dict(loader.stats, fallback=why)

    def padded(a):                                # engine.Model.__init__'s padding of a host array
        p = torch.zeros((a.shape[0], ld), dtype=torch.float32)
        p[:, :V] = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
        return p.to(dev)

    for name in names:
        if name in host:
            a = host[name]
            planes[name] = padded(a) if name.startswith('pmi') else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
            ranges[name] = (float(a.min()), float(a.max()))
    m.pmi, m.w1 = planes['pmi'], planes['pmi_w1']
    for name, attr in (('ed', 'edT'), ('ped', 'pedT')):
        p = torch.zeros((Vd, ld), dtype=torch.float32, device=dev)
        p[:, :V] = planes[name].t()
        setattr(m, attr, p)
    (pmin, pmax), (wmin, wmax) = ranges['pmi'], ranges['pmi_w1']
    m.frange = (pmin, pmax, wmin, wmax)
    m.ed_range = (ranges['ed'][1] - ranges['ed'][0], ranges['ped'][1] - ranges['ped'][0])
    return m
