#!/bin/bash
# Round-2 evidence run on one B200 (profiles/README.md): the default bench line, per-config bench
# lines, the ncu launch list of the default bench command, ncu --set full captures of the
# beam-search kernel for C2 (DRAM traffic -> profiles/k1_traffic.json), the hamming search and the
# PQ search, the flat search timing. Everything is written to OUTDIR.
# usage: scripts/profile_r02.sh OUTDIR
O=${1:?usage: scripts/profile_r02.sh OUTDIR}
mkdir -p "$O"
python bench.py > $O/bench_n1_r02.json 2> $O/bench_n1_r02.err
for w in c3 c4 c4cos c5b; do
  python bench.py --workload $w --extra none --steps 10 > $O/bench_${w}_r02.json 2> $O/bench_${w}_r02.err
done
python bench.py --workload c4 --points 10000000 --extra none --steps 5 --no-probe > $O/bench_c4_10m_r02.json 2> $O/bench_c4_10m_r02.err
python bench.py --workload c5a --steps 3 > $O/bench_c5a_r02.json 2> $O/bench_c5a_r02.err
SDB_FLAT_SKIP_EXACT=1 python scripts/bench_configs.py flat > $O/flat_r02.json 2> /dev/null
python scripts/flat_timeline.py --reps 7 --timeline --tag two-pass > $O/r02_flat_timeline.json 2> /dev/null
SDB_FLAT_LEVELS=1 python scripts/flat_timeline.py --reps 7 --tag "level scheme" > $O/r02_flat_levels.json 2> /dev/null
ncu --set full --clock-control none --import-source on -k regex:'tc5_filter|kth_thresh|rescore_warp' --launch-skip 8 -c 4 -f -o $O/prof_flat_r02 \
    python scripts/flat_timeline.py --reps 1 > $O/ncu_flat.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/launches_r02_bench.csv \
    python bench.py --steps 2 --warmup 1 > $O/ncu_bench_r02.log 2>&1
SDB_PROFILE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:beam_search -c 1 -f \
    -o $O/prof_k1_r02 python bench.py --graph gpu --extra none --steps 1 --no-probe --no-cpu-baseline > $O/ncu_k1_r02.log 2>&1
SDB_PROFILE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:beam_search -c 1 -f \
    -o $O/prof_k3fly_r02 python bench.py --workload c4 --points 300000 --extra none --steps 1 --no-probe > $O/ncu_k3fly_r02.log 2>&1
SDB_PROFILE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:beam_search -c 1 -f \
    -o $O/prof_k2_r02 python bench.py --workload c5b --points 2000000 --extra none --steps 1 --no-probe > $O/ncu_k2_r02.log 2>&1
ls -la $O/*.ncu-rep | tail -4
