# One GPU box, one call (`gpurun --timeout 3000 -- 'bash tools/gpu_round.sh'`): everything profiles/rNN_* is made of.
#   pytest -m gpu, bench lines of workloads B (headline), C, E, F, the ncu launch list of the bench command, one
#   `ncu --set full` capture of the step kernel in the steady-state workload (B, and F = the kernel with the convex
#   routines, late enough for the robots to have landed on the fields), the cycle
#   breakdown of workload F (timing variant: `make -C mjlab_b200/csrc variants` first), the
#   per-field parity table.  Outputs land in gpurun_out/ (merged back); copy what is to be kept into profiles/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm --format=csv > gpurun_out/smi.txt
timeout 1500 python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> gpurun_out/pytest_gpu.log
for w in B C E F; do timeout 300 python bench.py --workload $w > gpurun_out/bench_$w.json 2> gpurun_out/bench_$w.err; done
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file gpurun_out/launches.csv python bench.py --steps 2 --warmup 3 > gpurun_out/b_ncu.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:b2_step_kernel -s 245 -c 1 -f -o gpurun_out/step_kernel python tools/profile_step.py 4096 ncu > gpurun_out/ncu_full.log 2>&1
B2_WORKLOAD=F timeout 600 ncu --set full --clock-control none --import-source on -k regex:b2_step_kernel -s 1500 -c 1 -f -o gpurun_out/step_kernel_F python tools/profile_step.py 4096 ncu 200 > gpurun_out/ncu_full_F.log 2>&1
B2_WORKLOAD=F B2SIM_LIB=mjlab_b200/csrc/variants/libb2sim_timing.so timeout 300 python tools/phase_breakdown.py 4096 100 > gpurun_out/phase_F.txt 2>&1
for t in go1 g1 go1_rough g1_tracking; do B2_REF_TASK=$t B2_REF_DEVICE=cuda:0 timeout 300 python tests/ref_runner.py --rootdir /tmp tests/ref_env_cases.py > gpurun_out/ref_env_$t.log 2>&1; tail -1 gpurun_out/ref_env_$t.log; done  # the reference's own ManagerBasedRlEnv on libb2sim.so
for t in g1 go1_rough; do B2_REF_DEVICE=cuda:0 timeout 600 python tools/ref_env_bench.py $t 4096 50 2>&1 | tail -1 >> gpurun_out/ref_env_bench.txt; done; cat gpurun_out/ref_env_bench.txt  # the reference's env layer on this engine
timeout 900 python tools/parity_table.py 1024 > gpurun_out/parity_table.md 2> gpurun_out/parity_table.err
