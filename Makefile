# Builds libresr.so (sm_100a only) and the oracle helpers. `python -c "import __graft_entry__ as g; g.build()"` calls this.
NVCC      ?= nvcc
PKG       := real_esrgan-pytorch_b200
CSRC      := $(PKG)/csrc
LIB       := $(PKG)/lib/libresr.so
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr
SRCS      := $(wildcard $(CSRC)/*.cu)
OBJS      := $(patsubst $(CSRC)/%.cu,build/%.o,$(SRCS))
HDRS      := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/resr.h

all: $(LIB)

build/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	@mkdir -p $(PKG)/lib
	$(NVCC) -shared -o $@ $(OBJS) -cudart static

# development variants (same-box A/B through RESR_LIB_PATH, tools/ab.sh): make variant NAME=v1 [DEFS=-D...]
variant:
	@mkdir -p build/variants/$(NAME)
	for f in $(SRCS); do $(NVCC) $(NVFLAGS) $(DEFS) -c $$f -o build/variants/$(NAME)/$$(basename $$f .cu).o || exit 1; done
	$(NVCC) -shared -o build/variants/libresr_$(NAME).so build/variants/$(NAME)/*.o -cudart static

clean:
	rm -rf build $(LIB)

.PHONY: all clean variant
