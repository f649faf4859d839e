/* Minimal declarations of the Node-API (N-API v8) surface bbq_napi.c uses, so the shim can be
 * compile-checked in an image that has no Node headers (no node_api.h anywhere in this container).
 * On a machine with Node, build against the real <node_api.h> instead (-DBBQ_USE_REAL_NODE_API);
 * the names, argument orders and enum values below follow the published Node-API ABI. */
#ifndef BBQ_NODE_API_MIN_H
#define BBQ_NODE_API_MIN_H
#include <stddef.h>
#include <stdint.h>
#include <stdbool.h>
typedef struct napi_env__* napi_env;
typedef struct napi_value__* napi_value;
typedef struct napi_callback_info__* napi_callback_info;
typedef struct napi_ref__* napi_ref;
typedef enum { napi_ok = 0 } napi_status;
typedef enum { napi_int8_array, napi_uint8_array, napi_uint8_clamped_array, napi_int16_array, napi_uint16_array,
               napi_int32_array, napi_uint32_array, napi_float32_array, napi_float64_array } napi_typedarray_type;
typedef enum { napi_undefined, napi_null, napi_boolean, napi_number, napi_string, napi_symbol, napi_object,
               napi_function, napi_external, napi_bigint } napi_valuetype;
typedef napi_value (*napi_callback)(napi_env env, napi_callback_info info);
typedef void (*napi_finalize)(napi_env env, void* data, void* hint);
typedef struct { const char* utf8name; napi_value name; napi_callback method; napi_callback getter;
                 napi_callback setter; napi_value value; int attributes; void* data; } napi_property_descriptor;
napi_status napi_get_cb_info(napi_env, napi_callback_info, size_t* argc, napi_value* argv, napi_value* this_arg, void** data);
napi_status napi_typeof(napi_env, napi_value, napi_valuetype*);
napi_status napi_get_value_double(napi_env, napi_value, double*);
napi_status napi_get_value_int64(napi_env, napi_value, int64_t*);
napi_status napi_get_value_uint32(napi_env, napi_value, uint32_t*);
napi_status napi_get_value_external(napi_env, napi_value, void**);
napi_status napi_get_value_string_utf8(napi_env, napi_value, char* buf, size_t bufsize, size_t* result);
napi_status napi_get_typedarray_info(napi_env, napi_value, napi_typedarray_type*, size_t* length, void** data,
                                     napi_value* arraybuffer, size_t* byte_offset);
napi_status napi_create_external(napi_env, void* data, napi_finalize, void* hint, napi_value* result);
napi_status napi_create_arraybuffer(napi_env, size_t byte_length, void** data, napi_value* result);
napi_status napi_create_typedarray(napi_env, napi_typedarray_type, size_t length, napi_value arraybuffer,
                                   size_t byte_offset, napi_value* result);
napi_status napi_create_object(napi_env, napi_value* result);
napi_status napi_create_double(napi_env, double, napi_value* result);
napi_status napi_create_uint32(napi_env, uint32_t, napi_value* result);
napi_status napi_set_named_property(napi_env, napi_value object, const char* name, napi_value value);
napi_status napi_get_named_property(napi_env, napi_value object, const char* name, napi_value* result);
napi_status napi_define_properties(napi_env, napi_value object, size_t count, const napi_property_descriptor*);
napi_status napi_throw_error(napi_env, const char* code, const char* msg);
napi_status napi_get_undefined(napi_env, napi_value* result);
napi_status napi_create_reference(napi_env, napi_value value, uint32_t initial_refcount, napi_ref* result);
napi_status napi_delete_reference(napi_env, napi_ref ref);
#define NAPI_MODULE_INIT() napi_value napi_register_module_v1(napi_env env, napi_value exports)
#endif
