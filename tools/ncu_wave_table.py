"""Per-layer table of one full 37-slice wave of the convolution kernel from an `ncu --set full ... --page raw --csv` export of
`tools/conv_probe 37 2 1 0` (reps = 0: one launch per layer in network order):

    ncu --set full -k regex:conv_tc_kernel -c 21 -f -o wave tools/conv_probe 37 2 1 0
    ncu -i wave.ncu-rep --page raw --csv > wave_raw.csv
    python tools/ncu_wave_table.py wave_raw.csv profiles/r02_conv_wave_table.md profiles/r02_conv_traffic.json
"""
import csv
import json
import sys

UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-9, "us": 1e-6, "ms": 1e-3, "s": 1.0}
LAYERS = ["down0.block3", "down1.block0", "down1.block3", "down2.block0", "down2.block3", "down3.block0", "down3.block3",
          "down4.block0", "down4.block3", "up0.up1x1", "up0.block0", "up0.block3", "up1.up1x1", "up1.block0", "up1.block3",
          "up2.up1x1", "up2.block0", "up2.block3", "up3.up1x1", "up3.block0", "up3.block3+head"]
GFLOP = [4.832, 2.416, 4.832, 2.416, 4.832, 2.416, 4.832, 2.416, 4.832, 1.074, 9.664, 4.832, 1.074, 9.664, 4.832, 1.074, 9.664,
         4.832, 1.074, 9.664, 4.832 + 0.0252]
# algorithmic bytes per slice: split-plane activations in (4 B per value) + out (4 B per value, + pooled copy) ; weights excluded
def main():
    src, md_path, json_path = sys.argv[1:4]
    rows = list(csv.reader(open(src)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    ix = {h: i for i, h in enumerate(hdr)}

    def val(d, name):
        return float(d[ix[name]]) * UNIT.get(units[ix[name]], 1.0)

    out = ["# r02 — one 37-slice wave of `conv_tc_kernel` under `ncu --set full --clock-control none` (one launch per layer)", "",
           "Durations under ncu are cold-cache and serialised; the DRAM traffic per launch is what `bench.py` reports as",
           "`roofline.traffic` (mean over the 21 launches).  Algorithmic FLOPs: SURVEY.md section 8a x 37 slices.", "",
           "| layer | ms | algorithmic TFLOP/s | tensor pipe active % | tc smem reads % of peak | DRAM read MB | DRAM write MB | DRAM % of peak | L2 hit % |",
           "|---|---|---|---|---|---|---|---|---|"]
    traffic = []
    for i, d in enumerate(data[:21]):
        t = val(d, "gpu__time_duration.sum")
        rd, wr = val(d, "dram__bytes_read.sum"), val(d, "dram__bytes_write.sum")
        traffic.append(rd + wr)
        out.append("| %s | %.3f | %.0f | %.1f | %.1f | %.1f | %.1f | %.1f | %.1f |" % (
            LAYERS[i], t * 1e3, GFLOP[i] * 37 / t / 1e3, float(d[ix["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"]]),
            float(d[ix["l1tex__data_pipe_tc_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"]]) if "l1tex__data_pipe_tc_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed" in ix else float("nan"),
            rd / 1e6, wr / 1e6, float(d[ix["gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"]]), float(d[ix["lts__t_sector_hit_rate.pct"]])))
    mean = sum(traffic) / len(traffic)
    out += ["", "Mean DRAM traffic: **%.1f MB per launch** (%.2f GB per wave)." % (mean / 1e6, sum(traffic) / 1e9), ""]
    open(md_path, "w").write("\n".join(out) + "\n")
    json.dump({"mean_bytes_per_launch": mean, "launches": len(traffic), "per_layer_bytes": dict(zip(LAYERS, traffic)),
               "source": src}, open(json_path, "w"), indent=1)
    print("wrote", md_path, json_path, "mean %.1f MB" % (mean / 1e6))


if __name__ == "__main__":
    main()
