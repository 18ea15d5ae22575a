# ncu evidence for profiles/ (run on the GPU box: bash tools/prof_r2.sh [tag]).  Reports are summarised on the box
# (tools/ncu_summary.py, tools/ncu_src.py) and deleted: only text comes back through gpurun_out/ (64 MiB limit).
cd $GRAFT_REPO_ROOT
T=${1:-r2m}
O=gpurun_out
S="python bench.py --steps 2 --warmup 3 --no-cpu-baseline"
$S > $O/${T}_plain.log 2>&1 || exit 1
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/${T}_launches.csv $S > $O/${T}_ncu_launch.log 2>&1
python tools/ncu_summary.py launches $O/${T}_launches.csv $O/${T}_launches_summary.txt
SS="python bench.py --steps 1 --warmup 3 --no-cpu-baseline --rep-cpu 128"
$SS > $O/${T}_plain_small.log 2>&1 || exit 1
summ() { # report -> summary + per-opcode / stall table, then drop the report
  python tools/ncu_summary.py kernel $O/$1.ncu-rep $O/$1.txt
  ncu -i $O/$1.ncu-rep --page source --csv --print-source sass > /tmp/$1_src.csv 2>/dev/null
  python tools/ncu_src.py /tmp/$1_src.csv 12 >> $O/$1.txt 2>&1
  rm -f $O/$1.ncu-rep
}
for k in k1_up_mma k1_down_mma k2_tiles k2_paired k3_simulate; do
  ncu --set full --clock-control none --import-source on -k regex:$k -s 6 -c 1 -f -o $O/${T}_$k $SS > $O/${T}_ncu_$k.log 2>&1
  summ ${T}_$k
done
python tools/k4dbg.py > $O/${T}_k4_plain.log 2>&1 || exit 1
ncu --set full --clock-control none --import-source on -k regex:k4r_rounds -c 1 -f -o $O/${T}_k4r_rounds python tools/k4dbg.py > $O/${T}_ncu_k4r.log 2>&1
summ ${T}_k4r_rounds
tail -c 300 $O/${T}_plain.log
