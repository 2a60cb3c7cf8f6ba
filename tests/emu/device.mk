# TEST INFRASTRUCTURE ONLY: the host emulation (cg_emu.cpp) with the device-resident entry cg_process_device (cg_emu_device.cpp) as a
# shared library, for the CPU tests that call the emulated C ABI directly (tests/test_device_batch.py).  make -C tests/emu -f device.mk
CS := ../../crumble_b200/csrc
CFLAGS := -O2 -g -Wall -ffp-contract=off -DCG_EMU_CROSSCHECK -I$(CS)/hts_lite -I$(CS)
all: libcg_emu.so
libcg_emu.so: cg_emu_device.cpp cg_emu.cpp $(CS)/cg_host.cpp $(CS)/cg_params.c $(CS)/cg_pipeline.h $(CS)/cg_core.h $(CS)/cg_cells.h $(CS)/cg_column_lean.h ../../include/crumble_gpu.h
	gcc $(CFLAGS) -fPIC -c $(CS)/cg_params.c -o cp_pic.o
	g++ $(CFLAGS) -fPIC -shared -Wl,-Bsymbolic cg_emu_device.cpp $(CS)/cg_host.cpp cp_pic.o -o $@ -lm -lpthread
clean:
	rm -f cp_pic.o libcg_emu.so
.PHONY: all clean
