"""TEST DOUBLE for K8 (mlbp_parse_float_text, csrc/parse.cu): FakeKernels plus the text parser, emulated in Python on host
pointers.  Fields are split in Python and converted with float(); the placement, the checks, the state words and the list of
hard fields (more than 19 significant digits whose rounding the first 19 do not decide) are the kernel's.  Never imported by
the package."""
import re

import numpy as np

from fake_kernels import FakeKernels, _arr


class TextKernels(FakeKernels):
    """FakeKernels plus mlbp_parse_float_text"""

    def mlbp_parse_float_text(self, text, n_bytes, file_offset, n_cols, max_rows, out, ld_out, state, hard, hard_cap, tile_ws):
        if n_bytes == 0:
            return
        st = _arr(state, np.uint64, 8)
        data = bytes(_arr(text, np.uint8, n_bytes))
        O = _arr(out, np.float32, max_rows * ld_out) if max_rows else None
        H = _arr(hard, np.int64, 2 * hard_cap) if hard_cap else None
        num = re.compile(rb'[+-]?(?:(\d+)\.?(\d*)|\.(\d+))(?:[eE]([+-]?\d+))?')
        special = re.compile(rb'[+-]?(?:inf|infinity|nan)', re.IGNORECASE)
        errors, k = [], int(st[0])
        key = lambda b: (~b & 0xffffffffffffffff) if b >> 63 else b | (1 << 63)

        def record(off, kind):
            errors.append(((file_offset + off) << 3) | kind)

        pos = 0
        for line in data.split(b'\n'):
            for j, c in enumerate(line):
                ok = 0x20 <= c < 0x7f or c in b'\t\x0b\x0c' or (c == 13 and j == len(line) - 1 and pos + j + 1 < n_bytes)
                if not ok:
                    record(pos + j, 4)
                    break
            body = line.split(b'#', 1)[0]
            fields = [(m.start(), m.group()) for m in re.finditer(rb'[^ \t\x0b\x0c\r]+', body)]
            if fields and len(fields) != n_cols:
                record(pos + fields[0][0], 2)
            for start, f in fields:
                row, col = divmod(k, n_cols)
                if row >= max_rows:
                    record(pos + start, 3)
                elif special.fullmatch(f) or num.fullmatch(f):
                    m = num.fullmatch(f)
                    v = float(f)
                    if m:
                        intd, frac = (m.group(1), m.group(2)) if m.group(1) is not None else (b'', m.group(3))
                        sig = (intd + frac).lstrip(b'0')
                        if len(sig) > 19 and sig[19:].strip(b'0'):
                            # the kernel rounds from the first 19 digits w and from w + 1 and lists the field when they differ
                            w, q = int(sig[:19]), int(m.group(4) or 0) - len(frac) + len(sig) - 19
                            if float('%de%d' % (w, q)) != float('%de%d' % (w + 1, q)):
                                n = int(st[5])
                                st[5] = n + 1
                                if n < hard_cap:
                                    H[2 * n], H[2 * n + 1] = file_offset + pos + start, k
                                k += 1
                                continue
                    O[row * ld_out + col] = np.float32(v)
                    b = int(np.float64(v).view(np.uint64))
                    if v != v:
                        st[4] = int(st[4]) | (2 if b >> 63 else 1)
                    else:
                        kb = key(b)
                        st[2] = max(int(st[2]), ~kb & 0xffffffffffffffff)
                        st[3] = max(int(st[3]), kb)
                else:
                    record(pos + start, 1)
                k += 1
            pos += len(line) + 1
        st[0] = k
        if errors:
            st[1] = max(int(st[1]), ~min(errors) & 0xffffffffffffffff)
