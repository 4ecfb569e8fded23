"""Extract the equation tables the benchmark workloads are built from.

Run with VISYMRE_REFERENCE naming a checkout of the reference (aidalee123/Vision-SR):
    python tools/make_workload_tables.py
Writes vision-sr_b200/src/visymre/workloads/tables.json with, per table row, just what the
workload generator needs: name, formula string, variable names and sampling ranges.
Sources (reference scripts/): FeynmanEquations.xlsx (really an OLE2/BIFF8 .xls),
ode.xlsx (zip/XML), low_benchmarks.csv, low_benchmarks_scale.csv, and the 47-word
vocabulary pickled inside weights/meta/metadata.h5.
"""
import csv
import json
import os
import re
import struct
import sys
import zipfile
from xml.etree import ElementTree as ET

CHECKOUT = os.environ.get("VISYMRE_REFERENCE", "")
REF = os.path.join(CHECKOUT, "scripts")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "vision-sr_b200", "src", "visymre", "workloads", "tables.json")


# ---- OLE2 compound file + BIFF8 worksheet reader (just enough for one sheet) -------------
def _ole_stream(data, name):
    sec = 1 << struct.unpack_from("<H", data, 30)[0]
    n_fat = struct.unpack_from("<I", data, 44)[0]
    dir_start = struct.unpack_from("<I", data, 48)[0]
    difat = list(struct.unpack_from("<109I", data, 76))
    fat = []
    for s in difat[:n_fat]:
        fat += struct.unpack_from(f"<{sec // 4}I", data, 512 + s * sec)

    def chain(start):
        out, s = b"", start
        while s < 0xFFFFFFFC:
            out += data[512 + s * sec: 512 + (s + 1) * sec]
            s = fat[s]
        return out
    d = chain(dir_start)
    for i in range(0, len(d), 128):
        nlen = struct.unpack_from("<H", d, i + 64)[0]
        nm = d[i:i + max(nlen - 2, 0)].decode("utf-16-le", "ignore")
        if nm == name:
            start, size = struct.unpack_from("<I", d, i + 116)[0], struct.unpack_from("<I", d, i + 120)[0]
            return chain(start)[:size]
    raise KeyError(name)


def _rk(v):
    if v & 2:
        val = float(v >> 2 if not v & 0x80000000 else (v >> 2) - (1 << 30))
    else:
        val = struct.unpack("<d", struct.pack("<Q", (v & 0xFFFFFFFC) << 32))[0]
    return val / 100 if v & 1 else val


def read_xls(path):
    wb = _ole_stream(open(path, "rb").read(), "Workbook")
    pos, sst, cells, recs = 0, [], {}, []
    while pos + 4 <= len(wb):
        rid, ln = struct.unpack_from("<HH", wb, pos)
        recs.append((rid, wb[pos + 4: pos + 4 + ln]))
        pos += 4 + ln
    i = 0
    while i < len(recs):
        rid, body = recs[i]
        if rid == 0x00FC:  # SST, possibly continued
            chunks = [body]
            while i + 1 < len(recs) and recs[i + 1][0] == 0x003C:
                i += 1
                chunks.append(recs[i][1])
            n_unique = struct.unpack_from("<I", chunks[0], 4)[0]
            ci, off = 0, 8
            for _ in range(n_unique):
                buf = chunks[ci]
                if off >= len(buf):
                    ci, off = ci + 1, 0
                    buf = chunks[ci]
                nch, flags = struct.unpack_from("<HB", buf, off)
                off += 3
                rt = ext = 0
                if flags & 8:
                    rt = struct.unpack_from("<H", buf, off)[0]
                    off += 2
                if flags & 4:
                    ext = struct.unpack_from("<I", buf, off)[0]
                    off += 4
                s, wide = "", flags & 1
                while nch > 0:
                    buf = chunks[ci]
                    avail = (len(buf) - off) // (2 if wide else 1)
                    take = min(nch, avail)
                    raw = buf[off: off + take * (2 if wide else 1)]
                    s += raw.decode("utf-16-le" if wide else "latin-1")
                    off += len(raw)
                    nch -= take
                    if nch > 0:
                        ci, off = ci + 1, 1
                        wide = chunks[ci][0] & 1
                off += 4 * rt + ext
                sst.append(s)
        elif rid == 0x00FD:  # LABELSST
            r, c, _, idx = struct.unpack_from("<HHHI", body, 0)
            cells[(r, c)] = sst[idx]
        elif rid == 0x0203:  # NUMBER
            r, c, _ = struct.unpack_from("<HHH", body, 0)
            cells[(r, c)] = struct.unpack_from("<d", body, 6)[0]
        elif rid == 0x027E:  # RK
            r, c, _, v = struct.unpack_from("<HHHI", body, 0)
            cells[(r, c)] = _rk(v)
        elif rid == 0x00BD:  # MULRK
            r, c0 = struct.unpack_from("<HH", body, 0)
            n = (len(body) - 6) // 6
            for j in range(n):
                cells[(r, c0 + j)] = _rk(struct.unpack_from("<I", body, 4 + 6 * j + 2)[0])
        i += 1
    nrow = max(r for r, _ in cells) + 1
    ncol = max(c for _, c in cells) + 1
    return [[cells.get((r, c)) for c in range(ncol)] for r in range(nrow)]


def read_xlsx(path):
    z = zipfile.ZipFile(path)
    ns = {"m": "http://schemas.openxmlformats.org/spreadsheetml/2006/main"}
    shared = []
    if "xl/sharedStrings.xml" in z.namelist():
        for si in ET.fromstring(z.read("xl/sharedStrings.xml")).findall("m:si", ns):
            shared.append("".join(t.text or "" for t in si.iter("{%s}t" % ns["m"])))
    sheet = ET.fromstring(z.read("xl/worksheets/sheet1.xml"))
    rows = []
    for row in sheet.iter("{%s}row" % ns["m"]):
        vals = {}
        for c in row.findall("m:c", ns):
            col = re.match(r"[A-Z]+", c.get("r")).group(0)
            ci = 0
            for ch in col:
                ci = ci * 26 + ord(ch) - 64
            v = c.find("m:v", ns)
            if v is None:
                continue
            vals[ci - 1] = shared[int(v.text)] if c.get("t") == "s" else v.text
        rows.append([vals.get(i) for i in range(max(vals) + 1)] if vals else [])
    return rows


def main():
    out = {"generator": "tools/make_workload_tables.py", "source": "aidalee123/Vision-SR scripts/"}
    # Feynman
    rows = read_xls(os.path.join(REF, "FeynmanEquations.xlsx"))
    head = [str(h) for h in rows[0]]
    col = {h: i for i, h in enumerate(head)}
    feyn = []
    for r in rows[1:]:
        if not r[col["Filename"]] or not r[col["Formula"]]:
            continue
        nv = int(r[col["# variables"]])
        vs = []
        for i in range(1, nv + 1):
            lo, hi = r[col[f"v{i}_low"]], r[col[f"v{i}_high"]]
            if r[col[f"v{i}_name"]] is None:
                break
            # a few rows of the sheet carry no range: use the sheet's most common one
            vs.append(dict(name=str(r[col[f"v{i}_name"]]), low=float(lo) if lo is not None else 1.0,
                           high=float(hi) if hi is not None else 5.0))
        feyn.append(dict(name=str(r[col["Filename"]]), formula=str(r[col["Formula"]]),
                         replaced=str(r[col["replaced_formula"]]) if r[col.get("replaced_formula", 0)] else None,
                         variables=vs))
    out["feynman"] = feyn
    # ODE-Strogatz
    rows = read_xlsx(os.path.join(REF, "ode.xlsx"))
    out["ode"] = [dict(name=str(r[0]), formula=str(r[1])) for r in rows[1:] if r and r[0]]
    # low-dimensional benchmarks
    for key, fn in (("low", "low_benchmarks.csv"), ("low_scale", "low_benchmarks_scale.csv")):
        with open(os.path.join(REF, fn)) as fh:
            out[key] = [dict(name=r["name"], n_vars=int(r["variables"]), formula=r["expression"],
                             range=json.loads(r["range_"])) for r in csv.DictReader(fh)]
    # vocabulary
    sys.path.insert(0, CHECKOUT)
    import pickle
    import src.visymre.dclasses  # noqa: F401  (the pickle names this module)
    raw = open(os.path.join(REF, "weights/meta/metadata.h5"), "rb").read()
    md = pickle.loads(raw[2048:2048 + 2926])
    out["word2id"] = {k: int(v) for k, v in md.word2id.items()}
    out["total_variables"] = list(md.total_variables)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as fh:
        json.dump(out, fh, indent=0)
    print({k: (len(v) if isinstance(v, list) else type(v).__name__) for k, v in out.items()})
    print(feyn[0], feyn[-1], out["ode"][0], out["low"][0], sep="\n")


if __name__ == "__main__":
    main()
