# data collection: launch lists of the big configs, prefill launch list + ncu full of the mma cell
mkdir -p gpurun_out
timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none -c 500 --csv --log-file gpurun_out/launches_206M_B128.csv python bench.py --model 206M --envs 128 --domains mixed --steps 2 --warmup 1 --no-cpu-baseline --profile-steps 0 > gpurun_out/ncu_206.log 2>&1
timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_110M_B256.csv python bench.py --model 110M --envs 256 --discrete --steps 2 --warmup 1 --no-cpu-baseline --profile-steps 0 > gpurun_out/ncu_110.log 2>&1
timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_prefill_206M_B1.csv python tools/bench_prefill.py --model 206M --envs 1 --tokens 6000 --rollout 5 --check 0 --reps 1 > gpurun_out/ncu_pf.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:mlstm_cell_mma_kernel -s 3 -c 1 -o gpurun_out/prefill_cell_mma python tools/bench_prefill.py --model 206M --envs 1 --tokens 6000 --rollout 5 --check 0 --reps 1 > gpurun_out/ncu_pf2.log 2>&1
tail -3 gpurun_out/ncu_pf2.log
ls -la gpurun_out
