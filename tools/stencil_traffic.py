#!/usr/bin/env python3
"""DRAM traffic of ONE stencil launch from an ncu --set full capture -> profiles/r2_stencil_traffic.json (what bench.py's
roofline.traffic reads).  usage: tools/stencil_traffic.py REP.ncu-rep SOURCE_PIXELS OUT.json"""
import csv, io, json, subprocess, sys
rep, px, out = sys.argv[1], int(sys.argv[2]), sys.argv[3]
raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(raw))); hdr, units = rows[0], rows[1]
for r in rows[2:]:
    d = dict(zip(hdr, r))
    if "lsdb_stencil2_kernel" not in d.get("Kernel Name", ""):
        continue
    def val(k):
        v = float(d[k].replace(",", "")); u = units[hdr.index(k)].lower()
        return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[u]
    rd, wr = val("dram__bytes_read.sum"), val("dram__bytes_write.sum")
    json.dump({"kernel": d["Kernel Name"].split("(")[0], "dram_bytes": rd + wr, "dram_bytes_read": rd, "dram_bytes_write": wr, "source_pixels": px,
               "kernel_ms_under_ncu": float(d["gpu__time_duration.sum"].replace(",", "")) * {"ms": 1, "us": 1e-3, "ns": 1e-6, "s": 1e3}.get(units[hdr.index("gpu__time_duration.sum")].lower().replace("msecond", "ms").replace("usecond", "us").replace("nsecond", "ns").replace("second", "s"), 1),
               "from": f"{rep} (ncu --set full --clock-control none, one launch, {px} source pixels)"}, open(out, "w"), indent=1)
    print(open(out).read())
    break
