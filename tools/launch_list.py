"""ncu raw CSV (--metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --csv) of
tools/profile_forward.py -> compact per-launch list of the LAST forward + DRAM-traffic summary of the conv launches.

usage: python tools/launch_list.py gpurun_out/launches.csv profiles/r01_launches_s256_vNN.csv profiles/r01_conv_traffic_vNN.json
"""
import csv
import json
import re
import sys


def main():
    src, out_csv, out_json = sys.argv[1:4]
    rows = list(csv.reader(open(src, errors="replace")))
    h = next(i for i, r in enumerate(rows) if "Kernel Name" in r)
    hdr = rows[h]
    c = {k: hdr.index(k) for k in ("ID", "Kernel Name", "Grid Size", "Block Size", "Metric Name", "Metric Unit", "Metric Value")}
    launches = {}
    for r in rows[h + 1:]:
        if len(r) <= c["Metric Value"] or not r[c["ID"]].isdigit():
            continue
        k = int(r[c["ID"]])
        d = launches.setdefault(k, {"id": k, "kernel": r[c["Kernel Name"]], "grid": r[c["Grid Size"]], "block": r[c["Block Size"]]})
        v = float(r[c["Metric Value"]].replace(",", ""))
        unit = r[c["Metric Unit"]].lower()
        name = r[c["Metric Name"]]
        if name.startswith("gpu__time_duration"):
            d["time_us"] = v * {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(unit.replace("second", "s").replace("usecond", "us"), 1e-3)
        else:
            mult = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
            d["dram_read_bytes" if "read" in name else "dram_write_bytes"] = v * mult
    ls = [launches[k] for k in sorted(launches)]
    # last forward = from the last stem launch on
    stems = [i for i, d in enumerate(ls) if "stem_tc_kernel" in d["kernel"]]
    ls = ls[stems[-1]:]
    end = next((i for i, d in enumerate(ls) if "head_candidates" in d["kernel"] or "decode_kernel" in d["kernel"]), len(ls))
    fwd = ls[:end]

    def short(n):
        n = re.sub(r"\(anonymous namespace\)::|<unnamed>::|void ", "", n)
        n = re.sub(r"\((?:int)\)", "", n)
        return re.sub(r"\(.*\)$", "", n)

    with open(out_csv, "w") as f:
        f.write("# ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none "
                "<command> (launches from the last stem kernel on: one forward of the bench workload + whatever follows it)\n")
        w = csv.writer(f)
        w.writerow(["id", "kernel", "grid", "block", "time_us", "dram_read_bytes", "dram_write_bytes"])
        for d in ls:
            w.writerow([d["id"], short(d["kernel"]), d["grid"], d["block"], round(d.get("time_us", 0), 2), int(d.get("dram_read_bytes", 0)),
                        int(d.get("dram_write_bytes", 0))])
    conv = [d for d in fwd if "conv_tc_kernel" in d["kernel"]]
    tot = sum(d.get("dram_read_bytes", 0) + d.get("dram_write_bytes", 0) for d in conv)
    shares = {}
    for d in fwd:
        shares[short(d["kernel"])] = shares.get(short(d["kernel"]), 0) + d.get("time_us", 0)
    fwd_us = sum(d.get("time_us", 0) for d in fwd)
    js = {"source": out_csv, "streams": 256, "conv_launches": len(conv), "conv_time_us": sum(d.get("time_us", 0) for d in conv),
          "forward_time_us": fwd_us, "conv_share_of_forward": sum(d.get("time_us", 0) for d in conv) / fwd_us,
          "conv_dram_bytes_total": tot, "conv_dram_bytes_per_launch": tot / max(len(conv), 1),
          "time_us_by_kernel": {k: round(v, 1) for k, v in sorted(shares.items(), key=lambda kv: -kv[1])}}
    json.dump(js, open(out_json, "w"), indent=1)
    print(json.dumps(js, indent=1))


if __name__ == "__main__":
    main()
