#!/bin/bash
# GPU parity tests, phase profile, short bench (development helper).  Logs go to $OUT (default: a new temporary
# directory); the summary is printed.  Arguments go to pytest, e.g. -k "goldens or oracle_records or full_size" for a
# quick subset, --durations=8 for timings.
out=${OUT:-$(mktemp -d)}
mkdir -p "$out"
python -m pytest tests -m gpu -x -q "$@" 2>&1 | tail -25 > "$out/t.log"
python tools/phase_profile.py 64 > "$out/phase64.txt" 2>&1
python bench.py --no-cpu --no-ingest --steps 30 > "$out/bench_quick.json" 2> "$out/bench.err"
echo "logs in $out"; cat "$out/t.log" "$out/phase64.txt"; tail -3 "$out/bench.err"; python -c "
import json, sys; d=json.load(open(sys.argv[1])); print('units/s', d['value'], 'e2e', d['e2e']['value'], d['e2e_packed_masks']['value'], d['e2e_records_only']['value'], 'frac', d['roofline']['frac'])" "$out/bench_quick.json"
