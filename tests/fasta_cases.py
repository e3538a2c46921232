"""
FASTA files that exercise every rule of seq_sites.fasta_site_table (the host counter, the specification of the device
counter): line endings, whitespace, headers, case, IUPAC letters, sites cut by line, slab and sequence boundaries,
tip windows.  Used by tests/test_sites_cpu.py (the g++ build of sites.cuh) and tests/test_sites_gpu.py (the device).
"""
import gzip
import random

import numpy as np

from bin3c_b200 import seq_sites

ENZYMES = ['MluCI', 'Sau3AI']                   # AATT, GATC: dense four-cutters
LINE_WS = b'\t\x0b\x0c\x1c\x1d\x1e\x1f '         # str.strip() whitespace that does not end a line
EOLS = (b'\n', b'\r\n', b'\r')


def _seq_text(rng, n):
    """n bytes rich in AATT / GATC, with lower case, N and IUPAC letters, digits and gaps"""
    parts = [b'GATC', b'AATT', b'gatc', b'aatt', b'GA', b'TC', b'AAT', b'T', b'A', b'G', b'C', b'N', b'n', b'R', b'Y',
             b'-', b'*', b'0', b'x']
    out = b''
    while len(out) < n:
        out += rng.choice(parts)
    return out[:n]


def random_fasta(seed, n_records=12, wrap=None):
    """A seeded file mixing every line ending, blank and whitespace-only lines, leading, trailing and internal
    whitespace, '>' after whitespace, headers of every form, duplicates, text before the first header."""
    rng = random.Random(seed)
    eol = (lambda: rng.choice(EOLS))
    out = []
    if rng.random() < 0.5:
        out.append(b'text before the first header GATC' + eol())
    names = [b'c%d' % k for k in range(n_records)]
    for k in range(n_records):
        name = rng.choice(names[:k + 1])                        # duplicates
        form = rng.randrange(6)
        head = [b'>' + name, b'>', b'> ' + name, b'>\t' + name + b'\tdesc', b'>' + name + b' caf\xc3\xa9 long ' + b'd' * 90,
                b'>' + name + b'  '][form]
        out.append(head + eol())
        for _ in range(rng.randrange(5)):
            r = rng.random()
            if r < 0.15:
                out.append(eol())                               # blank line
            elif r < 0.25:
                out.append(bytes(rng.choice(LINE_WS) for _ in range(rng.randrange(1, 4))) + eol())
            elif r < 0.3:
                out.append(b'  >not a header GATC' + eol())
            else:
                lead = bytes(rng.choice(LINE_WS) for _ in range(rng.randrange(3))) if rng.random() < 0.4 else b''
                trail = bytes(rng.choice(LINE_WS) for _ in range(rng.randrange(3))) if rng.random() < 0.4 else b''
                body = _seq_text(rng, rng.randrange(0, wrap or 70))
                if rng.random() < 0.2 and len(body) > 2:
                    i = rng.randrange(1, len(body) - 1)
                    body = body[:i] + rng.choice([b' ', b'\t', b'  ']) + body[i:]
                out.append(lead + body + trail + eol())
    data = b''.join(out)
    if rng.random() < 0.4:
        data = data.rstrip(b'\r\n')                             # no final newline
    return data


def fixed_cases():
    """name -> file bytes"""
    c = {}
    c['lf'] = b'>a\nGATCAATT\nGATC\n>b\nAATTGATC\n'
    c['crlf'] = c['lf'].replace(b'\n', b'\r\n')
    c['cr'] = c['lf'].replace(b'\n', b'\r')
    c['mixed_no_final_eol'] = b'>a desc\r\nGAT\rCAA\nTT\r\n>b\rAATT\n\r\nGA\r\rTC\r\n\n\rGATC'
    c['cr_then_lf_lines'] = b'>a\r\rGATC\r\n\r\nGA\r\n\rTC\n\r>b\r\r\nAATT'
    c['whitespace'] = (b'>w\n\n   \n\t\x0b\x0c\x1c\x1d\x1e\x1f GA TC\x1f\x1e\x1d\x1c\x0c\x0b\t \nGATC GATC\n'
                       b'  \t  \n  >x GATC\nAA\tTT\n \x0bAATT\x0c \n')
    c['case_iupac'] = b'>l\ngatcAATTnnnGATCRYKMSWBDHVN\naattgAtCgAtC\n>m\nGANTCCTNAGRAATTY\n'
    c['straddle'] = b'>s\nGA\nTC\nA\nA\nT\nT\n>t\nTTAA\n>u\nGATCGA\n>v\nTCAATT'     # GA|TC across >v must not count
    c['headers'] = (b'>\nGATC\n> name\nAATT\n>\tx\ty\nGATC\n>n1 ' + b'desc ' * 40 + b'\nAATT\n>n2 caf\xc3\xa9\nGATC\n'
                    b'>n1\nGATCGATC\n>n2\n>last')
    c['pre_header'] = b'GATCGATC\nAATT\n>a\nGATC\n'
    c['empty'] = b''
    c['only_headers'] = b'>a\n>b\n>c'
    c['zero_length'] = b'>a\n>b\nGATC\n>c\n\n\n>d\n   \n>e\n'
    c['long_line'] = b'>big\n' + b'GATCAATTGC' * 1500 + b'\n>next\n' + b'AATT' * 3000
    c['long_header'] = b'>' + b'h' * 5000 + b' d\nGATC\n>' + b'g' * 9000 + b'\nAATTGATC'
    c['ws_run_across'] = b'>a\nGATC' + b' ' * 9000 + b'AATT\nGATC' + b'\t' * 9000 + b'\nAATT' + b' ' * 5000
    for s in range(6):
        c['random%d' % s] = random_fasta(100 + s)
    c['random_wide'] = random_fasta(7, n_records=30, wrap=300)
    return c


def tip_case(seed=3):
    """sequences of every length 0..40 made of AATT / GATC runs, so that sites sit on every window edge"""
    rng = random.Random(seed)
    out = []
    for n in range(41):
        body = _seq_text(rng, n).upper().replace(b'R', b'A')
        wrap = rng.choice([5, 7, 60])
        lines = [body[i:i + wrap] for i in range(0, len(body), wrap)] or [b'']
        out.append(b'>t%d\n' % n + b'\n'.join(lines) + b'\n')
    return b''.join(out)


def device_patterns(enzymes):
    """seq_sites' device pattern table for a list of enzymes"""
    return seq_sites._device_patterns(seq_sites._sites(enzymes))


def seeded_assembly(path, total_bp, seed=1, wrap=60, gz=False):
    """A seeded assembly of about total_bp bases: log-normal contig lengths (median ~20 kbp), ACGT with a few N runs,
    wrapped at `wrap` columns (None: one line per contig); gz: gzip level 1 (level 9 writes DNA at ~2 MB/s).  Returns
    the number of contigs."""
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b'ACGT', dtype=np.uint8)
    n, written = 0, 0
    with (gzip.open(path, 'wb', compresslevel=1) if gz else open(path, 'wb')) as f:
        while written < total_bp:
            ln = int(min(max(rng.lognormal(np.log(20000), 1.2), 200), 5_000_000))
            seq = lut[rng.integers(0, 4, ln)]
            if ln > 1000:
                at = int(rng.integers(0, ln - 100))
                seq[at:at + 100] = ord('N')
            f.write(b'>contig_%d len=%d\n' % (n, ln))
            body = seq.tobytes()
            if wrap:
                lines = np.frombuffer(body, dtype=np.uint8)
                full = ln // wrap * wrap
                block = np.concatenate([lines[:full].reshape(-1, wrap), np.full((full // wrap, 1), 10, np.uint8)],
                                       axis=1).tobytes()
                f.write(block + (body[full:] + b'\n' if ln > full else b''))
            else:
                f.write(body + b'\n')
            n += 1
            written += ln
    return n
