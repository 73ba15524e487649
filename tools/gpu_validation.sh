#!/usr/bin/env bash
# One gpurun call that regenerates the artefacts kept under profiles/ for the round's final code:
#
#   gpurun --timeout 1800 -- 'bash tools/gpu_validation.sh r02_final'
#
# (1) pytest -m gpu, (2) smoke(), (3) the default bench line (cfg3, all CPU legs) + builder lines for the other configs
# (cold and warm for the L2-resident ones), (4) the ncu launch list of the default bench command (device time of every
# launch: compare SHARES with the bench, not absolutes), (5) `ncu --set full` captures of the two stream kernels, (6) phase
# timings.  Outputs go to gpurun_out/<tag>_*; copy the ones to be judged into profiles/ (tools/ncu_extract.sh turns an
# .ncu-rep into the committed text extract).
set -u
TAG="${1:-rXX}"
OUT=gpurun_out
mkdir -p "$OUT"
python -m pytest tests -m gpu -q 2>&1 | tail -3 > "$OUT/${TAG}_pytest_gpu.txt"
cat "$OUT/${TAG}_pytest_gpu.txt"
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1 | tee "$OUT/${TAG}_smoke.txt"
python bench.py > "$OUT/${TAG}_bench_cfg3_n1.json" 2> "$OUT/${TAG}_bench_err.txt"
python - "$OUT/${TAG}_bench_cfg3_n1.json" <<'PY'
import json, sys
d = json.load(open(sys.argv[1]))
print("bench:", round(d["value"], 1), d["unit"], "|", round(d["ms_per_step"], 3), "ms/step | stream kernel", round(d["roofline"]["kernel_ms"], 3), "ms =",
      round(100 * d["roofline"]["frac"], 1), "% of", d["roofline"]["peak"], d["roofline"]["unit"], "| e2e", round(d["e2e"]["value"], 1), "| parity", d.get("parity_at_size"), "| clocks", d["clocks"])
PY
python bench.py --workload cfg3 --emulate-world 8 --steps 100 --no-cpu-baseline > "$OUT/${TAG}_bench_cfg3_shard8of8.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg2 --steps 500 --warmup 20 --no-nuts > "$OUT/${TAG}_bench_cfg2_n1.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg2 --steps 200 --warmup 20 --flush-l2 --no-cpu-baseline > "$OUT/${TAG}_bench_cfg2_n1_cold.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg1 --steps 300 --warmup 20 --no-nuts > "$OUT/${TAG}_bench_cfg1_n1.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg1 --steps 200 --warmup 20 --flush-l2 --no-cpu-baseline > "$OUT/${TAG}_bench_cfg1_n1_cold.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg5 --steps 50 --no-nuts > "$OUT/${TAG}_bench_cfg5_n1.json" 2>> "$OUT/${TAG}_bench_err.txt"
python bench.py --workload cfg4 --steps 5 --warmup 3 --no-cpu-baseline > "$OUT/${TAG}_bench_cfg4_n1.json" 2>> "$OUT/${TAG}_bench_err.txt"
for f in cfg3_shard8of8 cfg2_n1 cfg2_n1_cold cfg1_n1 cfg1_n1_cold cfg5_n1 cfg4_n1; do
python - "$OUT/${TAG}_bench_$f.json" $f <<'PY'
import json, sys
try:
    d = json.load(open(sys.argv[1]))
    print(sys.argv[2], round(d["value"], 1), d["unit"], round(d["ms_per_step"], 4), "ms/step kernel", round(d["roofline"]["kernel_ms"], 4), "frac", round(d["roofline"]["frac"], 4), "parity", (d.get("parity_at_size") or {}).get("rel_grad"))
except Exception as e:
    print(sys.argv[2], "FAILED", e)
PY
done
# plan build on the device: the builder's own kernels (key, CUB radix sort passes, bounds, rates, fill) with their device times,
# and gwi_model_create with a device-resident catalog (nothing crosses PCIe)
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"pd_|RadixSort" -c 40 --csv --log-file "$OUT/${TAG}_cfg3_plan_build_launches.csv" \
    python bench.py --steps 1 --warmup 3 --no-cpu-baseline > /dev/null 2> "$OUT/${TAG}_ncu_plan_err.txt"
GWI_PLAN_TIMING=1 python bench.py --steps 20 --no-cpu-baseline --catalog-on-device 2> "$OUT/${TAG}_plan_on_device_catalog_err.txt" | python -c "
import json,sys; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('cfg3 device-resident catalog: setup', d['setup_s'], 'log_l', d['result']['log_l'])" | tee "$OUT/${TAG}_plan_on_device_catalog.txt"
grep "gwi plan" "$OUT/${TAG}_plan_on_device_catalog_err.txt" | tail -1 | tee -a "$OUT/${TAG}_plan_on_device_catalog.txt"
# launch list of the default command (short run: ncu serialises and replays)
ncu --metrics gpu__time_duration.sum --clock-control none -s 40 -c 60 --csv --log-file "$OUT/${TAG}_cfg3_launches.csv" \
    python bench.py --steps 4 --warmup 3 --no-cpu-baseline > /dev/null 2> "$OUT/${TAG}_ncu_launches_err.txt"
# full captures: the headline kernel (one-role, cfg3) and the CTA-cooperative kernel on cfg2
ncu --set full --clock-control none --import-source on -k regex:stream_kernel -s 3 -c 1 -f -o "$OUT/${TAG}_cfg3_stream_kernel" \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2> "$OUT/${TAG}_ncu_full_err.txt"
# (the CTA-cooperative kernel runs the small catalogs: below 2.4e6 samples and chain batches; shards of cfg3 use the one-role kernel)
ncu --set full --clock-control none --import-source on -k regex:stream_cta_kernel -s 3 -c 1 -f -o "$OUT/${TAG}_cfg2_stream_cta_kernel" \
    python bench.py --workload cfg2 --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2>> "$OUT/${TAG}_ncu_full_err.txt"
for w in "cfg3" "cfg3 --emulate-world 8" "cfg2 --steps 300 --warmup 20" "cfg5"; do
  echo "== $w" >> "$OUT/${TAG}_phases.txt"
  GWI_PHASE_TIMING=1 python bench.py --no-cpu-baseline --workload $w 2>&1 >/dev/null | grep "gwi phases" >> "$OUT/${TAG}_phases.txt"
done
cat "$OUT/${TAG}_phases.txt"
ls -la "$OUT" | grep "${TAG}" | tail -30
