OUT=gpurun_out/r2cl
mkdir -p $OUT
timeout 500 ncu --set full --clock-control none --import-source on -k regex:k_hs_stream -s 1 -c 1 -o $OUT/hs_stream python tools/hector_stream_ncu.py 300 fast > $OUT/ncu_hs.log 2>&1
tail -3 $OUT/ncu_hs.log
if [ -f $OUT/hs_stream.ncu-rep ]; then
  ncu -i $OUT/hs_stream.ncu-rep --page raw --csv > $OUT/hs_stream_raw.csv 2>/dev/null
  ncu -i $OUT/hs_stream.ncu-rep --page source --print-source sass --csv > $OUT/hs_stream_source_sass.csv 2>/dev/null
  gzip -f $OUT/hs_stream_source_sass.csv
  ls -la $OUT/hs_stream.ncu-rep
  [ $(stat -c %s $OUT/hs_stream.ncu-rep) -gt 30000000 ] && rm -f $OUT/hs_stream.ncu-rep
fi
ls -la $OUT
