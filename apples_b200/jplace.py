"""jplace assembly (host).  Mirrors apples/jutil.py:1-19 (join_jplace) and the tail of run_apples.py:106-118."""
import gc
import json
import sys


def join_jplace(lst):
    """Merge per-query dicts into one.  Same quirk as jutil.py:11-19: with a single result an unplaceable query
    (edge_num == -1) empties the list; with several, the FIRST result is kept even if its edge_num is -1 and later
    unplaceable ones are dropped."""
    result = lst[0]
    if len(lst) == 1:
        if result['placements'][0]['p'][0][0] == -1:
            result['placements'] = []
        return result
    merged = list(result['placements'])
    for item in lst[1:]:
        if item['placements'][0]['p'][0][0] != -1:
            merged.extend(item['placements'])
    result['placements'] = merged
    return result


def assemble(results, extended_newick_string, argv=None):
    """run_apples.py:106-110"""
    result = join_jplace(results)
    result['tree'] = extended_newick_string
    result['metadata'] = {'invocation': ' '.join(sys.argv if argv is None else argv)}
    result['fields'] = ['edge_num', 'likelihood', 'like_weight_ratio', 'distal_length', 'pendant_length']
    result['version'] = 3
    return result


_REC = ('        {\n            "n": [\n                %s\n            ],\n            "p": [\n                [\n'
        '                    %s,\n                    %s,\n                    %s,\n                    %s,\n'
        '                    %s\n                ]\n            ]\n        }')
_INF = float('inf')


def _num(x):
    """One JSON number exactly as json.dumps writes it (float.__repr__, NaN / Infinity spelled out)."""
    if isinstance(x, float):
        if x != x:
            return 'NaN'
        if x == _INF:
            return 'Infinity'
        if x == -_INF:
            return '-Infinity'
        return float.__repr__(x)
    if isinstance(x, int) and not isinstance(x, bool):
        return int.__repr__(x)
    return json.dumps(x)


def dumps(result):
    """`json.dumps(result, sort_keys=True, indent=4)` (run_apples.py:114,117), byte for byte, without the pure-Python
    indenting encoder: the million placement records of a large run are written from one template (18 s -> 6 s per
    million queries).  Anything that does not look like an assembled jplace dict goes through json.dumps itself."""
    gc_was_on = gc.isenabled()
    gc.disable()  # millions of live records: a collection during the loop walks all of them
    try:
        placements = result['placements']
        if (not isinstance(placements, list) or not placements
                or any(type(k) is not str for k in result) or 'placements' not in result):
            raise ValueError
        recs = []
        esc = json.encoder.encode_basestring_ascii  # what json.dumps uses for str (ensure_ascii=True)
        fr = float.__repr__
        for pl in placements:
            if len(pl) != 2:
                raise ValueError
            n, p = pl['n'], pl['p']
            if len(n) != 1 or len(p) != 1 or type(n[0]) is not str:
                raise ValueError
            a, b, c, d, e = p[0]
            if (type(a) is int and type(b) is float and type(c) is int and type(d) is float and type(e) is float
                    and b - b == 0.0 and d - d == 0.0 and e - e == 0.0):  # the common record: finite floats
                recs.append(_REC % (esc(n[0]), a, fr(b), c, fr(d), fr(e)))
            else:
                recs.append(_REC % (esc(n[0]), _num(a), _num(b), _num(c), _num(d), _num(e)))
        body = '[\n' + ',\n'.join(recs) + '\n    ]'
        marker = '"@@APPLES_B200_PLACEMENTS@@"'
        shell = dict(result)
        shell['placements'] = marker[1:-1]
        text = json.dumps(shell, sort_keys=True, indent=4)
        if text.count(marker) != 1:
            raise ValueError
        return text.replace(marker, body)
    except (ValueError, KeyError, TypeError):
        return json.dumps(result, sort_keys=True, indent=4)
    finally:
        if gc_was_on:
            gc.enable()


def write_arrays(output_fp, names, in_backbone, out, extended_newick_string, exclude_intplace=False, argv=None, threads=0,
                 name_blob=None, name_off=None, alt=None):
    """The fast path of run_apples.py's tail (join_jplace + json.dumps + write, run_apples.py:106-118) straight from the
    device result arrays, without a million per-query dicts: the native writer (apples_jplace_write, hostio.cpp) renders
    the "placements" list, Python renders the few lines around it.  Output is byte-identical to
    `write(assemble(results_to_jplace(...)))`.  `names` is a list of str, or pass the reader's NUL-separated UTF-8 blob
    and offsets (FastaMatrix) as name_blob / name_off.  alt: the ranked records of place_*(keep > 1), written as
    results_to_jplace(..., alt=alt) lists them (apples_jplace_write_k).  Returns the number of placements written."""
    import ctypes as C
    import numpy as np
    from . import _lib
    lib = _lib.load()
    edge, error, distal, pendant, status = [np.ascontiguousarray(a) for a in out]
    n = int(edge.shape[0])
    if name_blob is None:
        enc = [s.encode('utf-8') for s in names]
        name_off = np.zeros(n + 1, np.int64)
        if n:
            np.cumsum([len(b) + 1 for b in enc], out=name_off[1:])
        name_blob = b'\0'.join(enc) + b'\0'
    name_off = np.ascontiguousarray(name_off, dtype=np.int64)
    inb = np.ascontiguousarray(np.asarray(in_backbone, dtype=np.uint8))
    marker = '@@APPLES_B200_PLACEMENTS@@'
    shell = {'placements': marker, 'tree': extended_newick_string,
             'metadata': {'invocation': ' '.join(sys.argv if argv is None else argv)},
             'fields': ['edge_num', 'likelihood', 'like_weight_ratio', 'distal_length', 'pendant_length'], 'version': 3}
    text = json.dumps(shell, sort_keys=True, indent=4)
    head, _, tail = text.partition('"' + marker + '"')
    err = C.create_string_buffer(512)
    nw = C.c_int64(0)
    blob = C.create_string_buffer(name_blob, len(name_blob)) if not isinstance(name_blob, C.Array) else name_blob
    args = (str(output_fp).encode(), head.encode(), (tail + '\n').encode(), n, C.cast(blob, C.c_void_p), _lib.ptr(name_off),
            _lib.ptr(inb), _lib.ptr(edge), _lib.ptr(error), _lib.ptr(distal), _lib.ptr(pendant), _lib.ptr(status),
            1 if exclude_intplace else 0)
    if alt is None:
        rc = lib.apples_jplace_write(*args, int(threads), C.byref(nw), err, 512)
    else:
        alt = [np.ascontiguousarray(a) for a in alt]
        keep = int(alt[1].shape[1])
        if any(a.shape[:1] != (n,) for a in alt) or any(a.shape[1:] != (keep,) for a in alt[1:]):
            raise ValueError('write_arrays: the ranked records do not match the %d placements' % n)
        rc = lib.apples_jplace_write_k(*args, keep, *[_lib.ptr(a) for a in alt], int(threads), C.byref(nw), err, 512)
    if rc != 0:
        raise OSError('writing %s failed: %s' % (output_fp, err.value.decode(errors='replace')))
    return int(nw.value)


def write(result, output_fp=None):
    """run_apples.py:112-118"""
    f = open(output_fp, 'w') if output_fp else sys.stdout
    f.write(dumps(result))
    f.write('\n')
    if output_fp:
        f.close()
