mkdir -p gpurun_out
python scripts/prof_kernels.py > gpurun_out/prof_plain.log 2>&1 || { tail -5 gpurun_out/prof_plain.log; exit 1; }
prof() {  # name regex which
  ncu --set full --clock-control none --import-source on -k regex:"$2" -s 1 -c 1 \
      -o gpurun_out/prof_$1_r1 python scripts/prof_kernels.py $3 > gpurun_out/ncu_$1.log 2>&1
  tail -1 gpurun_out/ncu_$1.log
}
prof tiles nr_tiles tiles
prof stream nr_stream stream
prof gridlj grid_logjoint grid
prof gridpost grid_posterior2 grid
prof gibbs gibbs_mvn_kernel gibbs
prof dmma mvn_logpdf_mma gibbs
ls -la gpurun_out/*.ncu-rep; du -sh gpurun_out
