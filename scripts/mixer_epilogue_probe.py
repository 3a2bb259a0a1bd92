import os, sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mixer_unit_timing as m
m.run("fp16x2", 64, 1376, "none")
m.run("fp16x2", 64, 1376, "gelu")
m.run("fp16x2", 344, 1376, "none")
m.run("fp16x2", 1376, 1376, "none")
