# final same-box tables of round 2: attention (ours fwd v5 / bwd vs cuDNN SDPA), GEMM vs cuBLAS, sweeps
timeout 300 python tools/attn_fwd_perf.py bwd sdpa > gpurun_out/r2_final_attention.txt 2>&1; echo "attn rc=$?"
timeout 300 python tools/gemm_vs_cublas.py > gpurun_out/r2_final_gemm_vs_cublas.txt 2>&1; echo "gemm rc=$?"
timeout 500 python tools/sweeps.py > gpurun_out/r2_final_sweeps.txt 2>&1; echo "sweeps rc=$?"
timeout 120 python tools/ew_perf.py > gpurun_out/r2_final_ew_perf.txt 2>&1; echo "ew rc=$?"
