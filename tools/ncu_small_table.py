"""Table of the forward's / pre-processing's small kernels from an `ncu --set full ... --page raw --csv` export of the bench
command itself (LM_GRAPHS=0, first launches of each kernel):

    LM_GRAPHS=0 ncu --set full -k regex:'stem_kernel|upsample2x|bodymask|resize_kernel' -c 12 -f -o small \
        python bench.py --steps 1 --warmup 0
    ncu -i small.ncu-rep --page raw --csv > small_raw.csv
    python tools/ncu_small_table.py small_raw.csv profiles/r02_call11_small_kernels.md "<title>" [hbm_peak_gbs]
"""
import csv
import sys

UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-9, "us": 1e-6, "ms": 1e-3, "s": 1.0}


def main():
    src, dst, title = sys.argv[1:4]
    peak = float(sys.argv[4]) if len(sys.argv) > 4 else 6567.1
    rows = list(csv.reader(open(src)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    ix = {h: i for i, h in enumerate(hdr)}

    def val(d, name):
        return float(d[ix[name]].replace(",", "")) * UNIT.get(units[ix[name]], 1.0)

    out = ["# " + title, "",
           "`ncu --set full --clock-control none` on `python bench.py --steps 1 --warmup 0` (LM_GRAPHS=0), the first launches of each kernel:",
           "a 300-slice volume through the pre-processing, 37-slice waves through the forward.  HBM peak of this pool's B200: %.0f GB/s" % peak,
           "(MEASURED_PEAKS.json).  Durations under ncu are cold-cache and serialised.", "",
           "| kernel | grid | ms | DRAM read MB | DRAM write MB | GB/s | of HBM peak | warps active % | issue active % | warp instr. (M) | regs |",
           "|---|---|---|---|---|---|---|---|---|---|---|"]
    for d in data:
        name = d[ix["Kernel Name"]].split("(")[0].split("::")[-1]
        t = val(d, "gpu__time_duration.sum")
        rd, wr = val(d, "dram__bytes_read.sum"), val(d, "dram__bytes_write.sum")
        gbs = (rd + wr) / t / 1e9
        out.append("| %s | %s | %.4f | %.1f | %.1f | %.0f | %.2f | %.1f | %.1f | %.1f | %s |" % (
            name, d[ix["launch__grid_size"]], t * 1e3, rd / 1e6, wr / 1e6, gbs, gbs / peak,
            float(d[ix["sm__warps_active.avg.pct_of_peak_sustained_active"]]),
            float(d[ix["smsp__issue_active.avg.pct"]]) if "smsp__issue_active.avg.pct" in ix else float(d[ix["smsp__issue_active.avg.pct_of_peak_sustained_active"]]),
            float(d[ix["smsp__inst_executed.sum"]].replace(",", "")) / 1e6, d[ix["launch__registers_per_thread"]]))
    open(dst, "w").write("\n".join(out) + "\n")
    print("\n".join(out))


if __name__ == "__main__":
    main()
