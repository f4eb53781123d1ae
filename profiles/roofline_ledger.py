"""Per-launch-class roofline ledger from a bench.py accounting file (the JSON that `bench.py --kernel-breakdown PATH` writes):
   for every tag (kernel class x layer geometry) the time the launch would take at the measured peaks,
   max(algorithmic bytes / HBM copy peak, FLOP / sustained bf16 peak), against the measured time.
usage: python profiles/roofline_ledger.py profiles/r02_kernel_breakdown_n1_b256_final.json [MEASURED_PEAKS.json] > profiles/r02_roofline_ledger.md"""
import json
import sys

src = sys.argv[1]
peaks = {"hbm_gbs": 6574.5, "bf16_tflops_sustained": 1472.2}
if len(sys.argv) > 2:
    peaks.update(json.load(open(sys.argv[2])))
hbm, tf = peaks["hbm_gbs"] * 1e9, peaks["bf16_tflops_sustained"] * 1e12
d = json.load(open(src))
rows, tot_ms, tot_floor = [], 0.0, 0.0
for v in d["by_tag"]:
    ms = v["ms"]
    t_mem, t_flop = v["bytes"] / hbm * 1e3, v["flop"] / tf * 1e3
    floor = max(t_mem, t_flop)
    tot_ms += ms
    tot_floor += floor
    rows.append((ms, v["tag"], v["n"], v["bytes"] / 1e9, v["flop"] / 1e12, "hbm" if t_mem >= t_flop else "tensor", floor))
rows.sort(reverse=True)
print("# Roofline ledger of one accounted step (%s)" % src)
print()
print("Peaks: HBM copy %.0f GB/s, sustained bf16 %.0f TFLOP/s (MEASURED_PEAKS.json).  floor = max(algorithmic bytes / HBM peak, FLOP / "
      "tensor peak) per class; launches without byte / FLOP accounting (spectral norm, Adam, tiny casts) have floor 0." % (hbm / 1e9, tf / 1e12))
print()
print("Sum of launch times %.1f ms; sum of floors %.1f ms = %.1f %% (the write-heavy 1x1 launches cannot reach the copy peak: write-only "
      "traffic tops out at 3.93 TB/s on this part, see profiles/r02_membw_probe.json)." % (tot_ms, tot_floor, 100 * tot_floor / tot_ms))
print()
print("| class / geometry | launches | ms | GB | TFLOP | bound | floor ms | floor / measured |")
print("|---|---|---|---|---|---|---|---|")
for ms, tag, n, gb, tflop, bound, floor in rows:
    if ms < 0.8:
        continue
    print("| %s | %d | %.2f | %.1f | %.2f | %s | %.2f | %.0f %% |" % (tag, n, ms, gb, tflop, bound if floor > 0 else "-", floor, 100 * floor / ms if ms else 0))
