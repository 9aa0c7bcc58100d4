/*
 * psx.h -- C ABI of libpsx.so: the B200 parameter-server data plane that stands
 * in for what douban/tfmesos reaches through tf.train.Server.
 *
 * The reference defines no FFI of its own for this path: it hands the process to
 * TensorFlow's distributed runtime at tfmesos/server.py:51-66 and the per-step
 * work (SURVEY.md 3.3) happens inside TF:
 *
 *   PULL   Variable -> _Send/_Recv, one RecvTensor per variable
 *          (triggered at examples/mnist/mnist.py:71, mnist_replica.py:204,
 *           matrix_factorization.py:45-49)
 *   PUSH   gradient _Send/_Recv worker -> ps            (same call sites)
 *   APPLY  ApplyGradientDescent / ApplyAdam on the PS    (mnist.py:55,
 *          mnist_replica.py:147-157, matrix_factorization.py:39-41)
 *
 * Each entry point below names the reference interface it replaces.  All
 * functions use C linkage, plain pointers and sizes; no C++ exception crosses
 * the boundary and nothing calls exit().  Return value: 0 on success, a negative
 * PSX_E* code otherwise, with a thread-local message behind psx_last_error()
 * (the Python side raises RuntimeError(msg), the reference's error style at
 * tfmesos/scheduler.py:398).  Device pointers are raw CUDA device addresses
 * (torch.Tensor.data_ptr()); streams are cudaStream_t passed as void*
 * (torch.cuda.current_stream().cuda_stream); 0 = the legacy default stream.
 *
 * Threading / lifetime contract: the id tables are mutex-protected, so calls on
 * DIFFERENT ids may come from different threads (the in-graph example drives N
 * workers from N threads, examples/mnist/mnist.py:76-80).  Calls on the same id
 * must be ordered by the caller (normally by issuing them on one stream), and an
 * object must outlive every other object mapped from its handle in the same
 * process (destroy clients before the shard they opened).  No entry point
 * synchronises the host except the *_values / *_state accessors and destroy.
 *
 * There is no CPU fallback: without a CUDA device every compute entry point
 * fails with PSX_ECUDA.
 */
#ifndef PSX_H_
#define PSX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSX_ABI_VERSION 11

/* error codes */
#define PSX_OK 0
#define PSX_EINVAL (-1)   /* bad argument / unknown id                       */
#define PSX_ECUDA (-2)    /* CUDA runtime or driver error (message has it)    */
#define PSX_ENOMEM (-3)
#define PSX_ESTATE (-4)   /* call not valid in the object's current state     */
#define PSX_EABI (-5)     /* handle blob from another ABI version             */

/* optimizers (reference: mnist.py:55 / mnist_replica.py:147; the others are
 * TF 0.12's ApplyMomentum / ApplyAdagrad / ApplyRMSProp).  The shard layout
 * depends on the optimizer, so a handle blob only opens in a build of the same ABI.
 *   opt       hyper[4]                       PSX_M              PSX_V     initial M / V
 *   SGD       {lr, -, -, -}                  -                  -
 *   ADAM      {lr, beta1, beta2, epsilon}    m                  v         0 / 0
 *   MOMENTUM  {lr, momentum, -, -}           accum              -         0
 *   ADAGRAD   {lr, initial_accum, -, -}      accum              -         initial_accum (> 0)
 *   RMSPROP   {lr, decay, momentum, eps}     ms (rms)           mom       1 / 0
 * Only Adam keeps beta powers; the others advance global_step alone. */
#define PSX_OPT_SGD 0
#define PSX_OPT_ADAM 1
#define PSX_OPT_MOMENTUM 2
#define PSX_OPT_ADAGRAD 3
#define PSX_OPT_RMSPROP 4

/* update disciplines (SURVEY.md appendix A.4) */
#define PSX_MODE_ASYNC_ORDERED 0 /* each slot applied on its own, slot order  */
#define PSX_MODE_SUM 1           /* ((g0+g1)+g2)+... then one apply           */
#define PSX_MODE_SYNC_MEAN 2     /* sum / (float)count, one apply             */
                                 /* (SyncReplicasOptimizer, mnist_replica.py:148-154) */

/* element types on the wire / in caller buffers */
#define PSX_F32 0
#define PSX_BF16 1

/* psx_set_values / psx_get_values selector */
#define PSX_VAR 0
#define PSX_M 1
#define PSX_V 2
#define PSX_SLOT0 16 /* PSX_SLOT0 + s selects gradient slot s (as f32)      */

#define PSX_MAX_SLOTS 16
#define PSX_HANDLE_BYTES 128 /* opaque blob shipped over the rendez-vous socket
                                (tfmesos/utils.py:6-15 framing)              */

int psx_abi_version(void);
const char *psx_last_error(void);

/* Number of CUDA devices visible; 0 with PSX_ECUDA when there is none. */
int psx_device_count(int *out_n);

/* Bind the calling process to a device before anything else: creates the
 * primary context, resolves the stream-memop driver entry points.
 * Replaces: tf.train.Server(server_def) start-up, tfmesos/server.py:52-61. */
int psx_init(int device_ordinal);

/* Let `device` read/write memory that lives on `peer` (idempotent). */
int psx_enable_peer(int device, int peer);

/* ------------------------------------------------------------------ PS side */

/* Allocate one PS shard in HBM on `device`: a flat f32 bucket `var[nelem]`
 * (+ the optimizer's state arrays, stored beta powers, global_step) and `n_slots`
 * gradient landing slots of `wire_dtype`, plus the flag words the kernels
 * synchronise on.  hyper: see the optimizer table above; an unknown `opt` or an
 * Adagrad initial accumulator <= 0 fails with PSX_EINVAL.
 * Replaces: variables + slot variables created on /job:ps/task:k by
 * replica_device_setter (mnist.py:43-46, mnist_replica.py:116-134) and
 * tf.get_variable under tf.device (matrix_factorization.py:21-28). */
int psx_shard_create(int device, uint64_t nelem, int opt, const float *hyper,
                     int n_slots, int wire_dtype, uint64_t *out_id);
int psx_shard_destroy(uint64_t id);
/* Blob a worker passes to psx_shard_open (CUDA-IPC inside). */
int psx_shard_export(uint64_t id, void *out_handle);
int psx_shard_set_hyper(uint64_t id, const float *hyper);

/* Synchronous host copies for init / tests / checkpoint.
 * Replaces: init_op (mnist.py:59, mnist_replica.py:164), Variable.eval()
 * (matrix_factorization.py:49). */
int psx_set_values(uint64_t id, int which, const float *host, uint64_t off, uint64_t n);
int psx_get_values(uint64_t id, int which, float *host, uint64_t off, uint64_t n);
/* stored Adam powers, global_step, number of completed apply rounds */
int psx_get_state(uint64_t id, float *b1p, float *b2p, int64_t *step, uint32_t *apply_seq);
int psx_set_state(uint64_t id, float b1p, float b2p, int64_t step);

/* Fused reduce(slots) + optimizer update + beta-power / global_step update over the
 * whole shard.  If wait_seq != 0 the stream first waits (cuStreamWaitValue32,
 * no SM is held) until every slot in [first_slot, first_slot+count) has been
 * pushed with seq >= wait_seq.  On completion the shard's apply_seq is
 * incremented and mirrored into every registered client.
 * Replaces: ApplyGradientDescent / ApplyAdam + AdamOptimizer._finish +
 * global_step assign_add on the PS (mnist.py:55; mnist_replica.py:147,156-157),
 * and SyncReplicasOptimizer's aggregation (mnist_replica.py:148-154). */
int psx_apply(uint64_t id, int mode, int first_slot, int count, uint32_t wait_seq,
              void *stream);

/* The same over elements [elem_off, elem_off + elem_n) of the shard only (elem_off
 * a multiple of 4; elem_n = 0 means the whole shard).  finish = 0 keeps the round
 * open: the beta powers, global_step and apply_seq move only with the launch that
 * passes finish = 1.  For row-block data parallelism (each worker owns a block of
 * rows of an embedding-like variable and pushes / pulls only that block): one
 * psx_apply_range per block with that block's owner as the only slot.
 * Replaces: the sparse (IndexedSlices) flavour of the apply ops for dense blocks. */
int psx_apply_range(uint64_t id, int mode, int first_slot, int count, uint64_t elem_off,
                    uint64_t elem_n, int finish, uint32_t wait_seq, void *stream);

/* Only the waiting half of psx_apply / psx_round: make `stream` wait until slots
 * [first_slot, first_slot+count) carry seq >= wait_seq.  Lets a caller bracket
 * the kernel alone with CUDA events. */
int psx_wait_slots(uint64_t id, int first_slot, int count, uint32_t wait_seq, void *stream);

/* ------------------------------------------------------------- worker side */

/* Map a PS shard into this process for use from `device` as gradient slot
 * `slot`.  Same-process handles are mapped directly, others through CUDA IPC.
 * Replaces: tf.Session(target) attaching to the PS devices (mnist.py:65,
 * mnist_replica.py:183, matrix_factorization.py:68). */
int psx_shard_open(const void *handle, int device, int slot, uint64_t *out_id);
int psx_shard_close(uint64_t id);
/* Blob for psx_shard_register_client: lets the PS mirror apply_seq into this
 * worker's HBM so the worker's pull waits on local memory. */
int psx_client_export(uint64_t client_id, void *out_handle);
int psx_shard_register_client(uint64_t shard_id, int slot, const void *client_handle);
/* Detach worker `slot` again: drains the shard's device, then unmaps the
 * worker's client block, mailbox and bound buffers.  A worker asks its PS for
 * this BEFORE psx_shard_close frees the block (a tf.Session closing,
 * examples/mnist/mnist_replica.py:183-220: the PS keeps serving the others). */
int psx_shard_unregister_client(uint64_t shard_id, int slot);

/* PUSH: copy n gradient elements grad_dev[0..n) into elements [off, off+n) of
 * this client's slot in the PS shard's HBM (vectorised stores, straight over
 * NVLink when the shard is on another GPU), then publish `seq` in the slot's
 * flag word (fence.sys + system-scope store) unless seq == 0.  src_dtype: type of grad_dev.
 * Replaces: gradient _Send/_Recv worker->ps, one RecvTensor per variable. */
int psx_push(uint64_t client_id, const void *grad_dev, uint64_t off, uint64_t n,
             int src_dtype, uint32_t seq, void *stream);

/* PULL: copy var[off, off+n) from the PS shard into param_dev[0..n), cast to
 * out_dtype.  If wait_seq != 0 the stream first waits until the shard has
 * completed apply round wait_seq.
 * Replaces: Variable read _Send/_Recv ps->worker, one RecvTensor per variable. */
int psx_pull(uint64_t client_id, void *param_dev, uint64_t off, uint64_t n,
             int out_dtype, uint32_t wait_seq, void *stream);

/* Bucketed tensor lists (BASELINE config #4: ResNet-50's 161 tensors): describe
 * once which device tensor (dev_ptrs[i], n[i] f32 elements) lives at which
 * shard element offset (offs[i]); afterwards ONE launch pushes / pulls the whole
 * list.  use_tma = 1: chunks stream global -> shared -> global with bulk-async
 * (TMA) copies through a 4-stage shared-memory ring; 0: plain 128-bit
 * loads/stores over the same chunk table.  Tensors whose address or offset is
 * not 16-byte aligned are copied element-wise.  f32 wire format only.
 * Replaces: the per-variable RecvTensor RPCs of one sess.run (SURVEY.md 2.2). */
int psx_list_create(uint64_t client_id, const void *const *dev_ptrs, const uint64_t *offs,
                    const uint64_t *n, int count, uint64_t *out_list_id);
int psx_list_destroy(uint64_t list_id);
int psx_push_list(uint64_t list_id, uint32_t seq, int use_tma, void *stream);
int psx_pull_list(uint64_t list_id, uint32_t wait_seq, int use_tma, void *stream);

/* ---------------------------------------------- one-shot fused round (sync) */

/* Exportable device buffers (worker gradient / parameter staging the PS-side
 * fused kernel reads and writes over NVLink). */
int psx_buffer_create(int device, uint64_t nbytes, uint64_t *out_id, void **out_dev_ptr);
int psx_buffer_export(uint64_t id, void *out_handle);
int psx_buffer_destroy(uint64_t id);

/* Bind worker `slot`'s gradient and parameter buffers (elements of the shard's
 * wire dtype -- f32, or bf16 with an f32 master on the PS -- range
 * [elem_off, elem_off + padded shard nelem) of each) to a shard for psx_round. */
int psx_round_bind(uint64_t shard_id, int slot, const void *grad_buf_handle,
                   const void *param_buf_handle, uint64_t elem_off);

/* Worker: "my bound gradient buffer holds round `seq`" (fence.sys + system-scope store into the
 * shard's slot flag).  Worker: wait until apply round `seq` is done. */
int psx_signal(uint64_t client_id, uint32_t seq, void *stream);
int psx_wait_applied(uint64_t client_id, uint32_t seq, void *stream);

/* Counter-based rendez-vous for synchronous rounds with many shards (one stream
 * memop instead of one per slot / per shard):
 *   - every completed psx_push / psx_signal also bumps the shard's `arrivals`
 *     counter; psx_wait_arrivals makes the stream wait for arrivals >= target
 *     (target = round * n_workers when every worker signals once per round);
 *   - a worker's MAILBOX is a counter in its own HBM that every shard it is
 *     registered with bumps when an apply / round completes; psx_wait_mailbox
 *     waits for counter >= target (target = round * n_shards);
 *   - psx_signal_many publishes one worker's readiness to up to 64 shards in a
 *     single launch. */
int psx_signal_many(const uint64_t *client_ids, int n, uint32_t seq, void *stream);
int psx_wait_arrivals(uint64_t shard_id, uint32_t target, void *stream);
int psx_mailbox_create(int device, uint64_t *out_id);
int psx_mailbox_export(uint64_t id, void *out_handle);
int psx_mailbox_destroy(uint64_t id);
int psx_shard_register_mailbox(uint64_t shard_id, int slot, const void *mailbox_handle);
int psx_wait_mailbox(uint64_t id, uint32_t target, void *stream);

/* Counted (graph-replayable) form of the same rendez-vous: every wait compares
 * with a CONSTANT and the waiter takes what it waited for off the counter, so a
 * round is the same command sequence every time and can be replayed from a CUDA
 * graph (stream memops are graph nodes).
 *   psx_round_counted / psx_apply_counted: wait for arrivals >= count, launch;
 *       the kernel's first instruction subtracts `count` from the counter.
 *   psx_signal_counted: like psx_signal_many, but first takes `consume` (last
 *       round's n_shards) off the worker's mailbox.
 *   psx_mailbox_consume: the same subtraction as a 1-thread launch (staged path).
 * Wait for a round's completion with psx_wait_mailbox(id, n_shards). */
int psx_round_counted(uint64_t shard_id, int mode, int first_slot, int count, void *stream);
int psx_apply_counted(uint64_t id, int mode, int first_slot, int count, void *stream);
int psx_signal_counted(const uint64_t *client_ids, int n, uint32_t seq, uint64_t mailbox_id,
                       uint32_t consume, void *stream);
int psx_mailbox_consume(uint64_t id, uint32_t n, void *stream);
/* Synchronous: set the counter (prime it with n_shards so that the first counted
 * round consumes the same constant as every later one). */
int psx_mailbox_set(uint64_t id, uint32_t value);

/* ONE kernel on the PS GPU: gather the bound gradients straight from the
 * workers' HBM (peer loads), reduce in registers in slot order, apply
 * the optimizer to var/m/v in place, and scatter the new parameters into every
 * bound parameter buffer (peer stores) -- push + sum + apply + pull with no
 * staging copy.  Waits like psx_apply. */
int psx_round(uint64_t shard_id, int mode, int first_slot, int count, uint32_t wait_seq,
              void *stream);

/* --------------------------------- NVSwitch multicast (NVLS), experimental --- */

/* Single-process multicast buffers: one allocation per listed GPU, all bound to
 * one multicast object.  psx_mc_broadcast stores a device array into EVERY GPU's
 * copy with multimem.st (the broadcast-back leg of a pull); psx_mc_reduce reads
 * the SUM over all copies with multimem.ld_reduce (the switch adds -- its order
 * is not the slot order, so this is a tolerance-checked mode).  `member` indexes
 * the device list given at creation; ranges are 16-byte granular.  Measured on 2
 * GPUs only; psx_round does not use them (DESIGN.md section 6). */
int psx_nvls_supported(int device, int *out);
int psx_mc_create(const int *devices, int n, uint64_t nbytes, uint64_t *out_id);
int psx_mc_destroy(uint64_t id);
int psx_mc_ptrs(uint64_t id, int member, void **out_unicast, void **out_multicast,
                uint64_t *out_size);
int psx_mc_broadcast(uint64_t id, int member, const void *src_dev, uint64_t off_bytes,
                     uint64_t nbytes, void *stream);
int psx_mc_reduce(uint64_t id, int member, void *dst_dev, uint64_t off_bytes, uint64_t nbytes,
                  void *stream);

/* ----------------------------------------- request-free serving (async) --- */

/* The reference's DEFAULT discipline -- every worker's push applied when it
 * arrives, nobody waits for anybody (examples/mnist/mnist_replica.py:198-205,
 * examples/mnist/mnist.py:63-72) -- without a host request per step.
 * psx_serve_start gives the shard a serving loop: one host thread polls the
 * shard's arrival counter (a 4-byte copy on the shard's own stream) and launches
 * [k_pick] [k_apply over the picked slots] whenever pushes have arrived; after 64
 * empty polls in a row it sleeps idle_sleep_us between polls (0 = keep spinning).
 * (No stream is ever left blocked in a wait-value for work that has not been
 * submitted yet: streams of a process share a few hardware channels.)
 *   mode PSX_MODE_ASYNC_ORDERED: every unconsumed push found by a pick is applied
 *     on its own (own beta powers, one global_step each), picks in arrival order,
 *     slots of one pick in slot order; the worker's client block receives the
 *     sequence number of its consumed push (psx_wait_applied) and the global_step
 *     that apply produced (psx_read_step_async).
 *   mode PSX_MODE_SYNC_MEAN: SyncReplicasOptimizer (mnist_replica.py:109-113,
 *     148-162) on the device: a push carries the global_step its parameters had
 *     (psx_push_stamped); older than the shard's global_step = stale = dropped;
 *     the first `replicas_to_aggregate` fresh ones BY ARRIVAL are averaged and
 *     applied once; then every registered worker gets a token (psx_wait_tokens),
 *     fast or slow, like the chief's token queue.
 * The host accessors (*_values, *_state, set_hyper, (un)register) pause the loop
 * for their duration; psx_shard_destroy stops it. */
int psx_serve_start(uint64_t shard_id, int mode, int replicas_to_aggregate, int idle_sleep_us);
int psx_serve_stop(uint64_t shard_id);
int psx_serve_stats(uint64_t shard_id, uint64_t *iterations, uint32_t *served, uint32_t *dropped,
                    int64_t *step);
/* psx_push that also records `stamp` (low 32 bits of the global_step the gradient
 * was computed at) for the sync serving mode. */
int psx_push_stamped(uint64_t client_id, const void *grad_dev, uint64_t off, uint64_t n,
                     int src_dtype, uint32_t seq, uint32_t stamp, void *stream);
/* Worker: the stream waits until this worker holds >= target tokens (one per
 * aggregated apply since the shard was created). */
int psx_wait_tokens(uint64_t client_id, uint32_t target, void *stream);
/* Host-side read of this worker's client block (sequence number of its last
 * consumed push, tokens, mirrored global_step) through a private stream; also
 * tells whether the shard lives in THIS process.  A process that serves a shard
 * itself must not stream-wait on it (psx_wait_applied / psx_wait_tokens refuse
 * with PSX_ESTATE: the wait would be submitted before the apply that satisfies
 * it and can deadlock behind a shared hardware channel) -- it polls with this. */
int psx_client_poll(uint64_t client_id, uint32_t *applied, uint32_t *tokens, int64_t *step,
                    int *in_process);
/* Worker: copy the global_step mirrored into this worker's client block by the
 * apply that consumed its last push into pinned host memory, asynchronously on
 * `stream` (the value sess.run([train_step, global_step]) returns,
 * mnist_replica.py:204) -- no host synchronisation. */
int psx_read_step_async(uint64_t client_id, int64_t *host_pinned, void *stream);

/* ------------------------------------------- index-list (sparse) rows --- */

/* IndexedSlices push for embedding-like variables (SURVEY.md 8f-3; what TF sends
 * for gather-based models instead of the dense gradient -- the reference's NMF
 * touches only row blocks of W, examples/matrix_factorization.py:21-28,43-49).
 * The shard is viewed as a [nelem / row_len, row_len] matrix.  psx_push_rows
 * copies k rows (rows_dev, k x row_len, src_dtype) and their row indices
 * (idx_dev, int64, STRICTLY ASCENDING -- the worker de-duplicates its own slices)
 * into this worker's landing slot and publishes `seq` like psx_push.
 * psx_apply_rows waits for the slots like psx_apply, merges rows pushed by
 * several workers in worker order (binary search, no float atomics: bit-
 * reproducible), divides by `count` for SYNC_MEAN, and applies the optimizer ONCE to
 * every touched row -- untouched rows keep var, m and v; beta powers and
 * global_step advance once per call. */
int psx_push_rows(uint64_t client_id, const int64_t *idx_dev, const void *rows_dev, uint64_t k,
                  uint64_t row_len, int src_dtype, uint32_t seq, void *stream);
int psx_apply_rows(uint64_t shard_id, int mode, int first_slot, int count, uint64_t row_len,
                   uint32_t wait_seq, void *stream);

/* Multi-process form (the product runs one process per GPU): one MEMBER per
 * (process, GPU).  The creator makes the multicast object for `n_devices`
 * members and gets its POSIX file descriptor, which the host ships to the other
 * processes over an AF_UNIX socket (SCM_RIGHTS -- the 128-byte blobs cannot carry
 * descriptors); they psx_mcx_import it.  Every member then adds its device
 * (psx_mcx_add_device), the host synchronises all members (barrier), and each
 * psx_mcx_bind creates this GPU's VMM allocation, binds it at offset 0 of the
 * object and maps it twice: at a unicast address (ordinary loads / stores) and,
 * as part of the whole team, at the multicast address.
 * Replaces the transport selection of tfmesos/scheduler.py:186 (protocol='grpc')
 * for the PS round's gather and broadcast-back legs. */
int psx_mcx_create(int device, int n_devices, uint64_t nbytes, int *out_fd, uint64_t *out_id);
int psx_mcx_import(int device, int n_devices, uint64_t nbytes, int fd, uint64_t *out_id);
int psx_mcx_add_device(uint64_t id);
int psx_mcx_bind(uint64_t id, void **out_unicast, void **out_multicast, uint64_t *out_size);
int psx_mcx_destroy(uint64_t id);

/* NVLS form of psx_round_bind: the workers' gradient / parameter tensors live at
 * byte offsets grad_off_bytes / param_off_bytes of every member's arena (same
 * layout in all of them); the shard covers elements [elem_off, elem_off + padded
 * nelem) of those tensors.  psx_round / psx_round_counted on a shard bound this
 * way gather with ONE multimem.ld_reduce.add.v4.f32 per vector (the switch sums
 * the n_members copies) and scatter with ONE multimem.st per vector; SUM and
 * SYNC_MEAN only, f32 wire, count must equal n_members.  Chosen once at set-up
 * (capability query psx_nvls_supported), never per call. */
int psx_round_bind_mc(uint64_t shard_id, uint64_t mcx_id, uint64_t grad_off_bytes,
                      uint64_t param_off_bytes, uint64_t elem_off, int n_members);

/* ------------------------------------------------------------- batching --- */

/* Several of the calls above in ONE crossing of the ABI, executed in order on
 * their own streams (a PS round is signal/push + wait + apply + wait/pull: five
 * calls whose host cost, not GPU time, bounds MNIST-sized rounds -- measured
 * 26 us/round at 64 KB).  Stops at the first failing op and returns its code;
 * *failed_index (may be NULL) receives its position. */
#define PSX_OP_PUSH 1          /* id=client ptr=grad off n a=src_dtype seq          */
#define PSX_OP_PULL 2          /* id=client ptr=param off n a=out_dtype seq=wait_seq */
#define PSX_OP_APPLY 3         /* id=shard a=mode b=first_slot c=count seq=wait_seq  */
#define PSX_OP_ROUND 4         /* id=shard a=mode b=first_slot c=count seq=wait_seq  */
#define PSX_OP_SIGNAL 5        /* id=client seq                                      */
#define PSX_OP_WAIT_APPLIED 6  /* id=client seq                                      */
#define PSX_OP_WAIT_SLOTS 7    /* id=shard b=first_slot c=count seq=wait_seq         */
#define PSX_OP_SIGNAL_MANY 8   /* ptr=uint64 client ids, n=count, seq                */
#define PSX_OP_WAIT_ARRIVALS 9 /* id=shard, waits for arrivals >= seq * c            */
#define PSX_OP_WAIT_MAILBOX 10 /* id=mailbox, waits for counter >= seq * c           */
#define PSX_OP_ROUND_COUNTED 11   /* id=shard a=mode b=first_slot c=count            */
#define PSX_OP_APPLY_COUNTED 12   /* id=shard a=mode b=first_slot c=count            */
#define PSX_OP_SIGNAL_COUNTED 13  /* ptr=client ids n=count id=mailbox c=consume seq  */
#define PSX_OP_MAILBOX_WAIT 14    /* id=mailbox, waits for counter >= c               */
#define PSX_OP_MAILBOX_CONSUME 15 /* id=mailbox, counter -= c                         */
typedef struct psx_op {
    int32_t op, a, b, c;
    uint64_t id, off, n;
    void *ptr;
    void *stream;
    uint32_t seq;
    uint32_t reserved;
} psx_op;
int psx_batch(const psx_op *ops, int n_ops, int *failed_index);

/* ------------------------------------------------------------ diagnostics */

/* Kernel launches issued by this library in this process since load. */
uint64_t psx_launch_count(void);
/* Raw device pointers (for zero-copy use by a co-resident worker and for
 * tests): which = PSX_VAR/PSX_M/PSX_V/PSX_SLOT0+s. */
int psx_shard_ptr(uint64_t id, int which, void **out_dev_ptr);
/* Plain device->device copy through the push kernel (bandwidth probes). */
int psx_copy(int device, void *dst, const void *src, uint64_t nbytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PSX_H_ */
