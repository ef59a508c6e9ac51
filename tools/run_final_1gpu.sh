# Round-end evidence on one B200: tests, both bench arms, per-view costs, ncu launch lists and one full capture.
T=${1:-r02}
M=gpu__time_duration.sum,smsp__inst_executed.sum,smsp__thread_inst_executed.sum,dram__bytes_read.sum,dram__bytes_write.sum
python -m pytest tests -m gpu -q 2>&1 | tail -4 | tee gpurun_out/${T}_pytest_tail.txt
python bench.py > gpurun_out/${T}_bench.json 2> gpurun_out/${T}_bench.err; tail -2 gpurun_out/${T}_bench.err
python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/${T}_bench_ref.json 2> gpurun_out/${T}_bench_ref.err
python tools/view_probe.py --grid --out gpurun_out/${T}_views.json > gpurun_out/${T}_views.log 2>&1; head -1 gpurun_out/${T}_views.log
for v in c2 gridworst eye12km zoom10; do
  ncu --metrics $M --clock-control none --csv --log-file gpurun_out/${T}_launch_$v.csv python tools/view_probe.py --ncu $v --reps 2 > /dev/null 2>&1
done
# the batch configuration bench.py times: one call of 256 panoramas = 4 chunks of 64 views x 46 kernels (the third call is listed)
ncu --metrics $M --clock-control none --csv --log-file gpurun_out/${T}_launch_batch256.csv python tools/batch_sweep.py --once 256 > /dev/null 2>&1
python tools/launch_table.py gpurun_out/${T}_launch_batch256.csv --last 184 --views 256 --json gpurun_out/${T}_batch_profile.json --source profiles/${T}_launch_batch256.csv | tail -12
# ... and the same for 256 distinct viewpoints (16x16 grid over the central degree: the C5 workload)
ncu --metrics $M --clock-control none --csv --log-file gpurun_out/${T}_launch_grid256.csv python tools/batch_sweep.py --once 256 --grid --grid-size 16 > /dev/null 2>&1
python tools/launch_table.py gpurun_out/${T}_launch_grid256.csv --last 184 --views 256 | tail -12
# one full capture of the batch configuration's kernels (one chunk of 64 views: 46 kernels of the third call)
# (the report itself is ~70 MB, more than gpurun copies back: it stays in /tmp, its summary comes home)
ncu --set full --clock-control none --import-source on -k regex:"k_mesh|k_blocks|k_raster|k_tiles|k_big|k_resolve4|k_near|k_prepare" -s 368 -c 46 -o /tmp/${T}_batch_chain python tools/batch_sweep.py --once 256 > gpurun_out/${T}_ncu_full.log 2>&1
python tools/ncu_summary.py /tmp/${T}_batch_chain.ncu-rep > gpurun_out/${T}_batch_chain_ncu_summary.txt 2>&1
python tools/batch_sweep.py --reps 4 --batches 16,64,256 --grid-size 16
ls -la gpurun_out | tail -20
