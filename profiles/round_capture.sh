#!/bin/bash
# One GPU-box pass that produces everything profiles/ tracks for a round: tests, bench (both arms),
# ncu launch list, ncu --set full captures of the dominant kernels, microbenchmarks.
#   usage (on the GPU box, from the repo root): bash profiles/round_capture.sh r02
tag=${1:-rXX}
out=gpurun_out
mkdir -p $out
timeout 400 python -m pytest tests -m gpu -x -q 2>&1 | tail -3 | tee $out/${tag}_pytest.txt
timeout 60 python -c "import __graft_entry__ as g; g.smoke(); print('SMOKE_OK')" 2>&1 | tail -2 | tee $out/${tag}_smoke.txt
timeout 400 python bench.py --steps 20 --warmup 5 2> $out/${tag}_bench.err | tail -1 > $out/${tag}_bench.json
timeout 300 python bench.py --impl reference --steps 20 --warmup 5 2>> $out/${tag}_bench.err | tail -1 > $out/${tag}_bench_reference.json
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 2000 --csv --log-file $out/${tag}_launches.csv python bench.py --steps 2 --warmup 3 --no-cpu > /dev/null 2>&1
python profiles/launch_shares.py $out/${tag}_launches.csv > $out/${tag}_launch_shares.txt 2>&1
for w in c2 c3 c4 c5 reduce; do
  k=k_filter_project; [ $w = c4 ] && k=k_hash_agg; [ $w = c5 ] && k=k_hash_agg; [ $w = reduce ] && k=k_reduce
  # c4 / c5: the second k_hash_agg launch of an operator pass is the bulk scan (the first is the 1 Mi-row prefix)
  skip=2; [ $w = c4 ] && skip=3; [ $w = c5 ] && skip=3
  timeout 200 ncu --set full --clock-control none --import-source on -k regex:$k -s $skip -c 1 -f -o /tmp/${tag}_$w python profiles/run_kernels.py $w > /dev/null 2>&1
  # summaries are made here: gpurun only brings back 64 MiB and one report is ~20 MiB
  python profiles/summarize.py /tmp/${tag}_$w.ncu-rep $out/${tag}_$w.summary.txt > /dev/null 2>&1
  python profiles/srcstat.py /tmp/${tag}_$w.ncu-rep 25 > $out/${tag}_$w.lines.txt 2>&1
done
cp /tmp/${tag}_c2.ncu-rep $out/ 2>/dev/null  # one raw report for auditing the summaries
timeout 120 python profiles/microbench_fp.py > $out/${tag}_microbench_fp.txt 2>&1
timeout 200 python profiles/microbench_agg.py > $out/${tag}_microbench_agg.txt 2>&1
./profiles/bin/scatter_ops2 > $out/${tag}_scatter_ops2.txt 2>&1
cat $out/${tag}_bench.json | head -c 1500; echo
tail -3 $out/${tag}_microbench_agg.txt
ls -la $out | grep ${tag}
