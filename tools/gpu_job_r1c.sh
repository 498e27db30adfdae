#!/bin/bash
# Round-1c evidence job (one B200): bench, per-format parity numbers, ncu launch list, ncu --set full of each hot kernel.
O=gpurun_out
python bench.py > $O/bench13.json 2> $O/bench13.err; echo "bench rc=$?"
python tools/probe_formats.py > $O/probe_formats.log 2>&1; echo "formats rc=$?"
ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file $O/r1c_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-graph --no-kernel-timing > $O/r1c_ncu_list.log 2>&1; echo "launch list rc=$?"
NCU="ncu --set full --clock-control none --import-source on -f"
$NCU -k regex:gemm2 -s 3 -c 1 -o $O/r1c_gemm_fc1_gelu python tools/prof_gemm_one.py 1536 384 gelu > $O/r1c_p1.log 2>&1; echo "p1 rc=$?"
$NCU -k regex:gemm2 -s 3 -c 1 -o $O/r1c_gemm_fc2_res python tools/prof_gemm_one.py 384 1536 res > $O/r1c_p2.log 2>&1; echo "p2 rc=$?"
$NCU -k regex:gemm2 -s 3 -c 1 -o $O/r1c_gemm_wgrad python tools/prof_gemm_one.py 1536 384 wgrad > $O/r1c_p3.log 2>&1; echo "p3 rc=$?"
$NCU -k regex:attn_fwd_sn -s 2 -c 1 -o $O/r1c_attn_fwd_sn python tools/prof_attn_one.py > $O/r1c_p4.log 2>&1; echo "p4 rc=$?"
$NCU -k regex:attn_bwd_sn -s 2 -c 1 -o $O/r1c_attn_bwd_sn python tools/prof_attn_one.py bwd > $O/r1c_p5.log 2>&1; echo "p5 rc=$?"
$NCU -k regex:ln_fwd -s 2 -c 1 -o $O/r1c_ln_fwd python tools/prof_elementwise_one.py ln_fwd > $O/r1c_p6.log 2>&1; echo "p6 rc=$?"
$NCU -k regex:ln_bwd -s 2 -c 1 -o $O/r1c_ln_bwd python tools/prof_elementwise_one.py ln_bwd > $O/r1c_p7.log 2>&1; echo "p7 rc=$?"
$NCU -k regex:quant_vec -s 2 -c 1 -o $O/r1c_quant python tools/prof_elementwise_one.py quant > $O/r1c_p8.log 2>&1; echo "p8 rc=$?"
$NCU -k regex:colsum -s 2 -c 1 -o $O/r1c_colsum python tools/prof_elementwise_one.py colsum > $O/r1c_p9.log 2>&1; echo "p9 rc=$?"
ls -la $O/*.ncu-rep | tail -12
