"""DRAM bytes per launch of every pipeline kernel from an `ncu --set full` capture (bench.py's roofline.traffic):
    python tools/ncu_traffic.py file.ncu-rep > profiles/rNN_traffic.json"""
import csv
import io
import json
import subprocess
import sys

NAMES = {"k_analyze_mad_rgba": "analyze_mad_fast", "k_band_list": "band_list", "k_mad_exact": "mad_exact", "k_plan": "plan",
         "k_shrink_tma": "resample_down", "k_shrink_warp": "resample_down_noslide", "k_expand_warp": "resample_up",
         "k_analyze_sobel_tma": "analyze_sobel"}
out = subprocess.run(["ncu", "-i", sys.argv[1], "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(out)))
h = rows[0]
ik, ir, iw = h.index("Kernel Name"), h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
units = rows[1]
scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
acc = {}
for r in rows[2:]:
    name = next((v for k, v in NAMES.items() if k in r[ik]), None)
    if name is None:
        continue
    b = float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]]
    acc.setdefault(name, []).append(b)
res = {k: int(sum(v) / len(v)) for k, v in acc.items()}
res["_source"] = ("ncu --set full --clock-control none, tools/prof_driver.py 3 (one synthetic 8K RGBA frame, second and third pass), "
                  "dram__bytes_read.sum + dram__bytes_write.sum per launch, mean")
print(json.dumps(res, indent=1))
