#!/usr/bin/env python3
"""Summarise an `ncu --set full` capture of one network pass of the tcgen05 conv family into profiles/*.json.

  python tools/ncu_conv_summary.py <capture>.ncu-rep profiles/r1_conv_ncu_full.json

The committed captures ran 4 network passes of 256 images (CFG-doubled n = 128) with 16 conv_tc launches each
(15 layers + the output conv) and kept `-s 16 -c 16`, exactly the second pass.  bench.py reads `traffic_bytes_per_pass`.
"""
import csv
import io
import json
import subprocess
import sys

LAYERS = ["down1.net.3", "ds1", "down2.net.0", "down2.net.3", "ds2", "mid.net.0", "mid.net.3", "attn.qkv", "attn.proj",
          "us2_conv", "up2.net.0", "up2.net.3", "us1_conv", "up1.net.0", "up1.net.3", "eps(out conv)"]


def num(d, key):
    v = d.get(key, "")
    try:
        return float(v.replace(",", ""))
    except ValueError:
        return None


def main():
    rep, out = sys.argv[1], sys.argv[2]
    note = sys.argv[3] if len(sys.argv) > 3 else ""
    images = int(sys.argv[4]) if len(sys.argv) > 4 else 256
    if rep.endswith(".csv.gz"):   # the `ncu -i ... --page raw --csv | gzip` dump of a capture
        import gzip
        raw = gzip.open(rep, "rt").read()
    else:
        raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True, check=True).stdout
    rows = list(csv.reader(io.StringIO(raw)))
    head, units, data = rows[0], rows[1], rows[2:]
    unit = dict(zip(head, units))
    global LAYERS
    tmac = [339.74, 151.00, 169.87, 339.74, 151.00, 84.93, 84.93, 28.31, 9.44, 339.74, 339.74, 84.93, 339.74, 679.48, 339.74]
    if len(data) == len(LAYERS) - 2:   # fused attention block build: attn.qkv / attn.proj are not conv_tc launches any more
        keep = [i for i, n in enumerate(LAYERS) if n not in ("attn.qkv", "attn.proj")]
        tmac = [tmac[i] for i in keep[:-1]]
        LAYERS = [LAYERS[i] for i in keep]
    if len(data) != len(LAYERS):
        raise SystemExit(f"expected {len(LAYERS)} conv_tc launches (one pass), the report holds {len(data)}")

    def scaled(d, key, to):
        v = num(d, key)
        if v is None:
            return None
        u = unit.get(key, "")
        mult = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(u) if to == "us" else \
            {"byte": 1e-6, "Kbyte": 1e-3, "Mbyte": 1.0, "Gbyte": 1e3}.get(u)
        return None if mult is None else v * mult

    layers, traffic = [], 0.0
    for name, row in zip(LAYERS, data):
        d = dict(zip(head, row))
        rd, wr = scaled(d, "dram__bytes_read.sum", "MB"), scaled(d, "dram__bytes_write.sum", "MB")
        e = {"layer": name, "kernel": d["Kernel Name"][:44],
             "us": round(scaled(d, "gpu__time_duration.sum", "us"), 3),
             "dram_read_MB": round(rd, 2), "dram_write_MB": round(wr, 2),
             "tensor_pipe_active_pct": num(d, "sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active")
             or num(d, "sm__inst_executed_pipe_tensor.avg.pct_of_peak_sustained_active"),
             "issue_active_pct": num(d, "smsp__issue_active.avg.pct_of_peak_sustained_active"),
             "lts_throughput_pct": num(d, "lts__throughput.avg.pct_of_peak_sustained_elapsed"),
             "grid": int(num(d, "launch__grid_size") or 0), "regs": int(num(d, "launch__registers_per_thread") or 0)}
        layers.append(e)
        if name != LAYERS[-1]:
            traffic += (rd + wr) * 1e6
    for e, m in zip(layers[:-1], tmac):
        e["tflops_under_ncu"] = round(2e6 * m * images / (e["us"] * 1e-6) / 1e12, 1)
    res = {"source": (note + "; " if note else "") + rep,
           "images_per_pass": images, "traffic_bytes_per_pass": traffic, "traffic_MB_per_image": traffic / images / 1e6,
           "conv_launches": len(layers) - 1,
           "conv_family_us": sum(e["us"] for e in layers[:-1]),
           "conv_family_tflops_under_ncu": 2e6 * sum(tmac) * images / (sum(e["us"] for e in layers[:-1]) * 1e-6) / 1e12,
           "algorithmic_MB_per_image_note": "inputs read once + outputs written once in bf16 = about 14.4 MB per image for "
                                            "these 15 layers; measured DRAM traffic is below that because part of every "
                                            "output is still in L2 when the kernel ends",
           "layers": layers[:-1], "eps_conv": layers[-1]}
    json.dump(res, open(out, "w"), indent=1)
    print(f"{out}: {sum(e['us'] for e in layers[:-1]):.1f} us for the {len(layers) - 1} layers, {traffic / images / 1e6:.2f} MB DRAM traffic per image")


if __name__ == "__main__":
    main()
