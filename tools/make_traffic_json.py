"""profiles/traffic.json (read by bench.py for `roofline.traffic`) from the ncu --set full summaries under profiles/."""
import csv
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROF = os.path.join(ROOT, "profiles")
# The inverse-dynamics captures (r2_rnea_f64_steady_ncu_full.csv, r1c_rnea_f32_ncu_full.csv) are of kernels that still loaded the
# gantry velocities (168 B / 84 B per sample); the current tau-only kernels move 144 B / 72 B.  They are left out until they are
# captured again, so bench.py reports roofline.traffic = null for that workload rather than a stale figure.
SOURCES = {
    "gram_f64_12500000": "r2_gram_v3_ncu_full.csv",
    "gram_f32_12500000": "r2_gram32_v3_ncu_full.csv",
    "linearize_f64_1048576": "r2_lin_final_ncu_full.csv",
}
UNIT = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}


def main():
    out, notes = {}, {}
    for key, fname in SOURCES.items():
        rows = {r[0]: r[1:] for r in csv.reader(open(os.path.join(PROF, fname)))}
        rd, wr = rows["dram__bytes_read.sum"], rows["dram__bytes_write.sum"]
        n = len(rd) - 1
        tot = [float(rd[1 + i]) * UNIT[rd[0]] + float(wr[1 + i]) * UNIT[wr[0]] for i in range(n)]
        out[key] = sum(tot) / n
        notes[key] = f"dram__bytes_read.sum + dram__bytes_write.sum, mean of {n} launch(es), profiles/{fname}"
    out["_source"] = notes
    out["_note"] = ("bytes per launch from ncu --set full (dram__bytes_read.sum + dram__bytes_write.sum).  No entry for the inverse-dynamics "
                    "workload: its captures predate the tau-only kernels (profiles/README.md)")
    with open(os.path.join(PROF, "traffic.json"), "w") as f:
        json.dump(out, f, indent=1)
    print({k: v for k, v in out.items() if not k.startswith("_")})


if __name__ == "__main__":
    main()
