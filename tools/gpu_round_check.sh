#!/usr/bin/env bash
# One gpurun call that re-validates the tree and collects every number / profile a round needs
# (a gpurun call costs 2-4 GPU-minutes of box time regardless of the command: bundle).
#
#   /usr/local/graft/bin/gpurun --timeout 1500 -- 'bash tools/gpu_round_check.sh r2'
#
# Outputs under gpurun_out/<tag>_*: pytest log, bench lines (own arm, reference arm), the ncu launch
# list of one fused pipeline run (durations + DRAM bytes), and `ncu --set full` reports of the
# kernels named in KERNELS (regex list).  Numbers printed under ncu are never bench values.
set -u
TAG=${1:-rN}
KERNELS=${KERNELS:-"cbca_win sgm_hpair sgm_pass stereo_join"}
OUT=gpurun_out
mkdir -p $OUT
date
python -m pytest tests -m gpu -q 2>&1 | tail -5 | tee $OUT/${TAG}_pytest.log
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -1
python tools/time_pipeline.py 2>&1 | tail -1
python tools/time_pipeline.py --exact 2>&1 | tail -1
python bench.py > $OUT/${TAG}_bench_n1.json 2> $OUT/${TAG}_bench_n1.err
cut -c1-220 $OUT/${TAG}_bench_n1.json
python bench.py --impl reference > $OUT/${TAG}_bench_reference_n1.json 2> /dev/null
cut -c1-120 $OUT/${TAG}_bench_reference_n1.json
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --csv \
    --log-file $OUT/${TAG}_launches_pipeline.csv python tools/run_op.py pipeline --iters 1 > /dev/null 2>&1
for k in $KERNELS; do
    timeout 300 ncu --set full --clock-control none --import-source on -k regex:"$k" -c 1 -f -o $OUT/${TAG}_prof_$k \
        python tools/run_op.py pipeline --iters 1 > /dev/null 2>&1
done
ls -la $OUT | grep ${TAG}_ | awk '{print $5, $9}'
echo finished
