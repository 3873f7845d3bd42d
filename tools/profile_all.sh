#!/bin/bash
# Round profiling pass (run under gpurun): bench without ncu first, then the ncu launch
# list of the same bench command, then one `--set full` capture per configuration's
# dominant kernel.  Reports land in gpurun_out/; tools/summarize_ncu.py turns them into
# the text summaries committed under profiles/.
set -u
O=gpurun_out
mkdir -p $O
python bench.py --steps 2 --warmup 3 > $O/bench_plain.json 2> $O/bench_plain.err || exit 1
ncu --metrics gpu__time_duration.sum --clock-control none -c 700 --csv --log-file $O/bench_launches.csv \
    python bench.py --steps 1 --warmup 1 > $O/bench_under_ncu.log 2>&1
NCU="ncu --set full --clock-control none --import-source on -c 1"
$NCU -k regex:k_pdm_v2_ws4 -s 2 -o $O/prof_pdm_v2_ws4 python tools/prof_pdm.py 131072 v2 > /dev/null 2>&1
$NCU -k regex:k_planar_tma -s 1 -o $O/prof_grain_tma python tools/prof_one.py grain 1 > /dev/null 2>&1
$NCU -k regex:k_interleaved4 -s 1 -o $O/prof_grain_il4 python tools/prof_one.py grain_il 1 > /dev/null 2>&1
$NCU -k regex:k_grain_mix3 -s 1 -o $O/prof_grain_mix3 python tools/prof_one.py gmix 1 > /dev/null 2>&1
$NCU -k regex:k_xvoice_mix -s 1 -o $O/prof_xvoice_mix python tools/prof_one.py xvoice 1 > /dev/null 2>&1
$NCU -k regex:k_voice_mix -s 1 -o $O/prof_voice_mix python tools/prof_one.py voice 1 > /dev/null 2>&1
$NCU -k regex:k_sweep_render -s 1 -o $O/prof_sweep_render python tools/prof_one.py sweep 1 > /dev/null 2>&1
$NCU -k regex:k_sweep_zsr_closed -s 1 -o $O/prof_sweep_zsr_closed python tools/prof_one.py sweep 1 > /dev/null 2>&1
$NCU -k regex:k_planar_tma -s 1 -o $O/prof_planar_tma python tools/prof_one.py pdmraw 1 planar_bulk=2 > /dev/null 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -c 12 --csv --log-file $O/launches_sweep.csv python tools/prof_one.py sweep 1 > /dev/null 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -c 12 --csv --log-file $O/launches_sweep_planar.csv python tools/prof_one.py sweep_planar 1 > /dev/null 2>&1
$NCU -k regex:graph_planar -s 1 -o $O/prof_graph_planar python tools/prof_one.py graph 1 > /dev/null 2>&1
ls -la $O/*.ncu-rep
# the reports together exceed what gpurun brings back: summarise here, keep only the headline report
SUMMARY_DIR=$O/summaries python tools/summarize_ncu.py $O/prof_*.ncu-rep
for f in $O/prof_*.ncu-rep; do case $f in *pdm_v2_ws4*) ;; *) rm -f $f ;; esac; done
du -sh $O
