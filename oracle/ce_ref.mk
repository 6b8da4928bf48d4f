# oracle/ce_ref.mk -- TEST INFRASTRUCTURE ONLY: the reference's own CE::EvalParallel (src/net/ce-loss.cc, already in
# REF_SRCS of oracle/Makefile) behind a small driver, oracle/ce_ref.cc, built from the same CPU objects:
#   make -C oracle -f ce_ref.mk ce     ->  oracle/_ref/ref_ce_cpu
# Only where the reference tree is present; elsewhere the tests replay the stored runs (tests/golden/runs).
include Makefile

ifneq ($(wildcard $(REF)/src/net/ce-loss.cc),)
ce: $(OUT)/ref_ce_cpu
else
ce:
	@echo "reference tree $(REF) not present: using prebuilt oracle/_ref binaries (if any)"
endif

$(OUT)/ref_ce_cpu: ce_ref.cc $(CPU_OBJS)
	$(CXX) $(REFFLAGS) ce_ref.cc $(CPU_OBJS) -o $@ $(LDCPU)

.PHONY: ce
