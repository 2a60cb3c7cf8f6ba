# TEST INFRASTRUCTURE ONLY: the host emulation with the device-resident entries (cg_emu_device.cpp) and the stream entry cg_stream_device
# (cg_emu_stream.cpp) as a shared library, for the CPU tests of streams (tests/test_device_stream.py).  make -C tests/emu -f stream.mk
CS := ../../crumble_b200/csrc
CFLAGS := -O2 -g -Wall -ffp-contract=off -DCG_EMU_CROSSCHECK -I$(CS)/hts_lite -I$(CS)
all: libcg_emu_stream.so
libcg_emu_stream.so: cg_emu_stream.cpp cg_emu_device.cpp cg_emu.cpp $(CS)/cg_host.cpp $(CS)/cg_params.c $(CS)/cg_pipeline.h $(CS)/cg_core.h $(CS)/cg_cells.h $(CS)/cg_column_lean.h ../../include/crumble_gpu.h
	gcc $(CFLAGS) -fPIC -c $(CS)/cg_params.c -o cps_pic.o
	g++ $(CFLAGS) -fPIC -shared -Wl,-Bsymbolic cg_emu_stream.cpp $(CS)/cg_host.cpp cps_pic.o -o $@ -lm -lpthread
clean:
	rm -f cps_pic.o libcg_emu_stream.so
.PHONY: all clean
