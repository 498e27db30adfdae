#!/bin/bash
# Round-2 evidence job (one B200): final bench, the reference arm, ncu launch list of the step, ncu --set full of the kernels
# that changed this round (each only after the same command has run clean without ncu).
O=gpurun_out
python bench.py > $O/r2_bench_final.json 2> $O/r2_bench_final.err; echo "bench rc=$?"
python bench.py --impl reference --steps 2 --warmup 1 > $O/r2_bench_ref.json 2> $O/r2_bench_ref.err; echo "ref rc=$?"
L="python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-graph --no-kernel-timing --no-quant-bench --no-configs"
$L > $O/r2_plain_list.log 2>&1 && ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file $O/r2_launches.csv $L > $O/r2_ncu_list.log 2>&1; echo "launch list rc=$?"
NCU="ncu --set full --clock-control none --import-source on -f"
python tools/prof_attn_one.py bwd > $O/r2_p1.log 2>&1 && $NCU -k regex:attn_bwd_sn -s 2 -c 1 -o $O/r2_attn_bwd_sn python tools/prof_attn_one.py bwd > $O/r2_p1n.log 2>&1; echo "attn bwd rc=$?"
$NCU -k regex:attn_fwd_sn -s 2 -c 1 -o $O/r2_attn_fwd_sn python tools/prof_attn_one.py bwd > $O/r2_p2n.log 2>&1; echo "attn fwd rc=$?"
python tools/prof_gemm_one.py 1536 384 dgelu > $O/r2_p3.log 2>&1 && $NCU -k regex:gemm2 -s 3 -c 1 -o $O/r2_gemm_dgelu python tools/prof_gemm_one.py 1536 384 dgelu > $O/r2_p3n.log 2>&1; echo "dgelu rc=$?"
python tools/prof_gemm_one.py 384 384 res > $O/r2_p4.log 2>&1 && $NCU -k regex:gemm2 -s 3 -c 1 -o $O/r2_gemm_proj_res python tools/prof_gemm_one.py 384 384 res > $O/r2_p4n.log 2>&1; echo "proj res rc=$?"
python tools/prof_gemm_one.py 1536 384 gelu > $O/r2_p5.log 2>&1 && $NCU -k regex:gemm2 -s 3 -c 1 -o $O/r2_gemm_gelu python tools/prof_gemm_one.py 1536 384 gelu > $O/r2_p5n.log 2>&1; echo "gelu rc=$?"
python tools/prof_segloss_one.py > $O/r2_p6.log 2>&1 && $NCU -k regex:upsample_ce -s 2 -c 1 -o $O/r2_segloss python tools/prof_segloss_one.py > $O/r2_p6n.log 2>&1; echo "segloss rc=$?"
python tools/prof_elementwise_one.py quant > $O/r2_p7.log 2>&1 && $NCU -k regex:quant_vec16 -s 1 -c 1 -o $O/r2_quant python tools/prof_elementwise_one.py quant > $O/r2_p7n.log 2>&1; echo "quant rc=$?"
